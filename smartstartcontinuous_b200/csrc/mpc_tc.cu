// mpc_tc.cu -- tcgen05 / TMEM rollout kernel for the random-shooting MPC (sm_100a only).
//
// Replaces the H sess.run float64 GEMM round trips of Dyn_Model.do_forward_sim
// (dynamics_model.py:204-240) + the numpy scoring of generate_scores_add_delta
// (NND_MB_agent.py:566-628) for the 2-hidden-layer dynamics MLP (the 2x500 network of the
// BASELINE configs).  Persistent CTA PAIRS (2-CTA clusters, tcgen05 cta_group::2): each CTA owns
// tiles of 128 sequences ("rows" = TMEM lanes) and walks them through all H steps without
// touching HBM for activations; the pair issues M = 256 MMAs so every weight byte streamed from
// L2 feeds two tiles -- each CTA holds only its half of every B tile, which halves the per-SM
// L2 -> shared-memory traffic that otherwise caps the kernel (~43 B/clk/SM chip-wide).
//
//   layer 1   [256 x K1] x [K1 x HP]   tcgen05.mma, A = split-bf16 input in smem (K1 = 16 or 32 slots),
//             B = W1 image (input, weights and bias are hi/lo bf16 splits packed along K, so the
//             layer is FP32-accurate although it runs on the tensor pipe); all HP/128 chunks are
//             issued back to back: odd chunks into the accumulator slots, even chunks into the
//             (then dead) H1 columns, converted in place
//   relu+cvt  TMEM accumulator chunk -> registers -> bf16x2 -> TMEM (becomes the A operand)
//   layer 2   [256 x HP] x [HP x HP]   tcgen05.mma kind::f16 (BF16 in, FP32 accumulate in TMEM),
//             A from TMEM, B = W2 streamed from L2 by the TMA engine (cp.async.bulk, pre-packed
//             32 KB core-matrix half blocks of 256 K elements) through a 4-stage mbarrier ring;
//             bias folded in via two constant-one hidden units (hi/lo split)
//   layer 3   fused into the layer-2 epilogue: relu, packed FP32 FFMA2 dot with W3 pairs from
//             shared memory
//   update    state += z * std_z + mean_z in FP32 registers; waypoint logic + progress/penalty
//             score (score.cuh) run in the shadow of the next step's layer-2 MMAs
//
// Warp roles per CTA: warps 0-7 = row warps (two threads per row: ch 0 feeds the network, ch 1
// scores; each takes half the columns of every accumulator chunk), warp 8 = MMA warp (leader CTA:
// issues every MMA of the pair, warp-uniform loop, one elected lane; peer CTA: relays "my half of
// the stage has landed" to the leader), warp 9 = TMA producer.
// TMEM per CTA (512 columns): [0,256) H1 as bf16 A operand, [256,512) 2-deep ring of 128x128 FP32
// accumulator chunks.  Two-tile schedule (PAIR, hp = 512, K1 = 16): two tiles per CTA half a step apart, each with
// H1 units 0-255 in TMEM and 256-511 in shared memory, so one tile's layer 2 covers the other's per-step chain.
// Cross-CTA signalling: mbarrier arrives on the leader's barriers
// (shared::cluster, release.cluster) and tcgen05.commit.cta_group::2 multicast to both CTAs.
#include <cuda_bf16.h>

#include <cstdlib>
#include <cstring>

#include "mpc_kernels.cuh"
#include "tc_ptx.cuh"
#include "tc_score_row.cuh"

namespace tc {

constexpr int TM = 128;                 // rows per tile (per CTA); the pair's MMA has M = 256
constexpr int NC = 128;                 // units per accumulator chunk (MMA N over the pair)
constexpr int NH = NC / 2;              // units of a chunk whose weights live in THIS CTA's smem
constexpr int KSLAB = 256;              // K elements per W2 stage (16 MMAs: amortises the issue loop)
constexpr int STAGE_BYTES = NH * KSLAB * 2;   // 32 KB per CTA and stage
constexpr int NSTAGE = 4;
constexpr int K1_MAX = 32;              // K slots of the layer-1 MMA: 16 (3 (dz + da) + 2 <= 16) or 32
constexpr int ACC_SLOTS = 2;
constexpr int W1_CHUNK_BYTES_MAX = NH * K1_MAX * 2;   // 4 KB per CTA and chunk
constexpr int A1_BYTES_MAX = TM * K1_MAX * 2;         // 8 KB
constexpr int ROW_WARPS = 8;                  // 2 threads per row: each takes half of the columns
constexpr int TPR = ROW_WARPS / 4;
constexpr int CPT = NC / TPR;                 // accumulator columns per thread and chunk
constexpr int ROW_THREADS = ROW_WARPS * 32;
constexpr int THREADS = ROW_THREADS + 64;
constexpr int HP_MAX = 512;
constexpr int MAX_DIN = (K1_MAX - 2) / 3;   // 3 slots per input + 2 bias slots <= K1
// layer-3 outputs computed for state dimension d, and the layer-1 input slots: state j -> input j
// (j < dz), action j -> input dz + j; three K slots per input + two bias slots
__host__ __device__ constexpr int dz_of(int d) { return d <= 2 ? 2 : (d <= 3 ? 3 : (d <= 4 ? 4 : 8)); }
__host__ __device__ constexpr int k1_slots(int d, int da) { return 3 * (dz_of(d) + da) + 2 <= 16 ? 16 : 32; }
__host__ __device__ constexpr int w3_pair_floats(int dz) { return dz <= 2 ? 4 : (dz <= 4 ? 8 : 16); }
constexpr uint32_t TMEM_COLS = 512;
constexpr uint32_t COL_H1 = 0, COL_ACC = 256;
constexpr int CLUSTER = 2;

struct Params {
    const __nv_bfloat16* w1_img;        // [2 (cta)][HP/128][4][64][8]
    const __nv_bfloat16* w2_img;        // [HP/128 (n)][HP/128 (k-slab)][2 (cta)][16][64][8]
    const float* w3;                    // [HP/2 (unit pairs)][DZP][2]: packed for FFMA2
    const float* b3;                    // [SS_MAX_D] output-layer bias (device memory: ss_dyn_commit rewrites it)
    int hp;                             // padded hidden width (multiple of 128)
    int din;
    long long tile_begin, tile_end;     // this launch rolls the tiles [tile_begin, tile_end) of the batch
    int iters;                          // tile iterations per CTA (same for all: pair lock-step)
    int pair_iters;                     // of these, iterations run two at a time (two-tile schedule)
    unsigned long long* prof;
};

// D f32, A/B bf16, K-major, N = 128, M = 256 (cta_group::2)
constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(NC >> 3) << 17) |
                           ((uint32_t)((2 * TM) >> 4) << 24);


#define TC_TRACE(ev)                                                                              \
    do {                                                                                          \
        if (p.prof && blockIdx.x == 0 && lane == 0 && trace_it == 0 && trace_t >= 10 && trace_t < 13) \
            trace_s[(trace_t - 10) * 256 + (ev)] = (unsigned long long)clock64();                  \
    } while (0)

// Two-tile schedule (PAIR): every CTA walks two tiles at once, offset by half a step.  TMEM holds K-slab 0
// (units 0-255) of both tiles' H1 ([0,128) tile 0, [128,256) tile 1) and the two accumulator slots; K-slab 1
// (units 256-511) of each tile's H1 is a K-major no-swizzle A image in shared memory.
// W2 ring of the two-tile schedule: 4 x 16 KB (half a K-slab per stage).  Two 32 KB stages leave one stage of
// lead, less than the latency of a 32 KB bulk copy from L2 at the 32 B/clk per SM that a busy tensor pipe consumes.
constexpr int PAIR_STAGES = 4;
constexpr int PSTAGE_BYTES = STAGE_BYTES / 2;
constexpr int H1S_BYTES = TM * (HP_MAX - KSLAB) * 2;              // 64 KB: one tile's K-slab 1
constexpr int PAIR_K1 = 16;                                       // layer-1 K slots the PAIR layout has room for
constexpr int PAIR_BARS = 2 * PAIR_STAGES + 2 * ACC_SLOTS + 7;
constexpr size_t SMEM_LIMIT = 232448;                             // 227 KiB of dynamic shared memory per CTA

// two-tile schedule: stamps of half-steps 20-25 (steps 10-12 of both tiles of block 0's first tile pair), 64 per
// half-step.  MMA warp: 2n+k before / 8+2n+k after the K-slab k of chunk n, 16 chunk-3 scratch free seen,
// 17 chunk 2 issued, 18 / 19 before / after the waits for the other tile's layer 1.  Row warps (ch 0 at +20, ch 1 at +40): 0 start,
// 1 other tile's step finished, 2 its x-split written, 3 scoring done, 4-6 epilogue n0-n2 done, 7 layer 1 converted.
#define PAIR_TRACE(hs_, ev)                                                                               \
    do {                                                                                                  \
        if (p.prof && blockIdx.x == 0 && lane == 0 && (hs_) >= 20 && (hs_) < 26 && (ev) < 64)             \
            trace_s[((hs_) - 20) * 64 + (ev)] = (unsigned long long)clock64();                            \
    } while (0)

template <int DZ, bool PAIR = false>
struct SmemT {
    // dynamic shared memory carve-up (offsets in bytes from a 128-byte aligned base)
    static constexpr size_t W2_RING = 0;
    static constexpr size_t W1 = W2_RING + (size_t)NSTAGE * STAGE_BYTES;
    static constexpr size_t A1 = W1 + (size_t)(HP_MAX / NC) * W1_CHUNK_BYTES_MAX;
    static constexpr size_t W3 = A1 + (size_t)A1_BYTES_MAX;
    static constexpr size_t ZX = W3 + (size_t)(HP_MAX / 2) * w3_pair_floats(DZ) * 4;
    static constexpr size_t BARS = ZX + (size_t)TPR * TM * 8 * 4;
    static constexpr int N_BARS = 3 * NSTAGE + 2 * ACC_SLOTS + 2 * (HP_MAX / NC) + 2;
    static constexpr size_t TMEM_PTR = BARS + (size_t)N_BARS * 8;
    static constexpr size_t TRACE = TMEM_PTR + 16;     // SS_TC_TRACE stamps (only when tracing)
    static constexpr size_t END = TRACE;
};
// Layout of the kernels that run the two-tile schedule (K1 = 16 only).  The one-tile ring of a trailing
// odd tile aliases the two H1 K-slab-1 images (the producer starts it only after the last two-tile MMA).
template <int DZ>
struct SmemT<DZ, true> {
    static constexpr size_t H1S = 0;                                                  // 2 x 64 KB
    static constexpr size_t W2_RING = 0;                                              // one-tile ring, 4 x 32 KB
    static constexpr size_t PRING = H1S + 2 * (size_t)H1S_BYTES;                      // two-tile ring, 4 x 16 KB
    static constexpr size_t W1 = PRING + (size_t)PAIR_STAGES * PSTAGE_BYTES;
    static constexpr size_t A1 = W1 + (size_t)(HP_MAX / NC) * NH * PAIR_K1 * 2;       // 8 KB of W1
    static constexpr size_t W3 = A1 + (size_t)TM * PAIR_K1 * 2;                       // one 4 KB A1 tile
    static constexpr size_t ZX = W3 + (size_t)(HP_MAX / 2) * w3_pair_floats(DZ) * 4;
    static constexpr size_t BARS = ZX + (size_t)TPR * TM * 8 * 4;
    static constexpr int N_BARS = SmemT<DZ, false>::N_BARS + PAIR_BARS;
    static constexpr size_t TMEM_PTR = BARS + (size_t)N_BARS * 8;
    static constexpr size_t TRACE = TMEM_PTR + 16;
    static constexpr size_t END = TRACE;
    static_assert(NSTAGE * STAGE_BYTES <= 2 * H1S_BYTES, "the one-tile ring fits in the H1 images");
    static_assert(END + 128 <= SMEM_LIMIT, "two-tile layout exceeds 227 KiB");
};
// (dz, K1) layouts whose two-tile layout fits: <4,2,16>, <4,3,16>.  <4,4,32> and <8,8,32> need 16 KB of W1 and
// an 8 KB A1 tile (and <8,8,32> a 16 KB W3): they keep the one-tile schedule.
__host__ __device__ constexpr bool pair_layout_fits(int dz, int k1) {
    return k1 == PAIR_K1 && dz <= 3;
}

// DT: register copies of the state (4 or 8); DZ: layer-3 outputs computed (>= d; 2, 3, 4 or 8), which is
// also where the action inputs start (action j -> input DZ + j); K1T: K slots of the layer-1 MMA (16 when
// 3 (DZ + da) + 2 <= 16, else 32).  DZ and K1T must be the dz_of / k1_slots the images were packed with
// (ctx tc_dz / tc_k1): the launcher dispatches on exactly that pair, and every (d, da) that
// mpc_tc_shape_supported accepts has an instantiation -- <4,2,16>, <4,2,32>, <4,3,16>, <4,3,32>,
// <4,4,32>, <8,8,32> (tests/test_gpu_mpc_dims.py runs each against the float64 oracle).
// ROWS: every sequence starts at its own row of a.state0_rows (load_start, forward simulation).
// PAIR: the first 2 * p.pair_iters tile iterations run on the two-tile schedule (pair_layout_fits, hp = 512),
// the rest on the one-tile schedule.
template <int DT, int DZ, int K1T, bool ROWS = false, bool PAIR = false>
__global__ void __launch_bounds__(THREADS, 1) mpc_rollout_tc_kernel(const RolloutArgs a, const Params p) {
    pdl_trigger();      // the reduce / tail kernels behind this launch may be scheduled (they wait for its completion)
    extern __shared__ __align__(128) unsigned char smem[];
    using Smem = SmemT<DZ, PAIR>;
    static_assert(!PAIR || pair_layout_fits(DZ, K1T), "no two-tile layout for this instantiation");
    constexpr int MAXIN = (K1T - 2) / 3;            // network inputs the A tile has slots for
    constexpr int W1_CHUNK_BYTES = NH * K1T * 2;
    constexpr int DZP = w3_pair_floats(DZ) / 2;     // layer-3 outputs padded to 2 / 4 / 8
    unsigned char* w2_ring = smem + Smem::W2_RING;
    unsigned char* w1s = smem + Smem::W1;
    unsigned char* a1s = smem + Smem::A1;
    float* w3s = reinterpret_cast<float*>(smem + Smem::W3);
    float* zx = reinterpret_cast<float*>(smem + Smem::ZX);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Smem::BARS);
    uint64_t* w2_full = bars;                           // local: this CTA's half of the stage has landed
    uint64_t* w2_peer = w2_full + NSTAGE;               // leader's copy: the peer's half has landed
    uint64_t* w2_empty = w2_peer + NSTAGE;              // local: the pair's MMAs are done with the stage
    uint64_t* acc_full = w2_empty + NSTAGE;             // local: accumulator chunk complete (commit)
    uint64_t* acc_free = acc_full + ACC_SLOTS;          // leader's copy: both CTAs' row warps drained it
    uint64_t* h1_ready = acc_free + ACC_SLOTS;          // leader's copy [HP_MAX / NC]
    uint64_t* l1_full = h1_ready + HP_MAX / NC;         // local: layer-1 chunk complete (commit)
    uint64_t* x_ready = l1_full + HP_MAX / NC;          // leader's copy
    uint64_t* w1_full = x_ready + 1;                    // local
    // two-tile schedule (PAIR): its own barriers, so the one-tile phases start fresh after it
    uint64_t* p_w2_full = w1_full + 1;                  // [PAIR_STAGES] as w2_full
    uint64_t* p_w2_empty = p_w2_full + PAIR_STAGES;     // [PAIR_STAGES] as w2_empty
    uint64_t* p_acc_full = p_w2_empty + PAIR_STAGES;    // [ACC_SLOTS] layer-2 chunk complete
    uint64_t* p_acc_free = p_acc_full + ACC_SLOTS;      // [ACC_SLOTS] leader's copy: slot drained (layer 2 or layer-1 chunk 1)
    uint64_t* p_x_ready = p_acc_free + ACC_SLOTS;       // leader's copy: a tile's layer-1 A tile is in smem
    uint64_t* p_l1a = p_x_ready + 1;                    // local: layer-1 chunks 0-2 of a tile complete
    uint64_t* p_l1b = p_l1a + 1;                        // local: layer-1 chunk 3 complete
    uint64_t* p_scr = p_l1b + 1;                        // leader's copy: chunk 2 loaded, its scratch columns are free
    uint64_t* p_h1t = p_scr + 1;                        // leader's copy: H1 K-slab 0 (TMEM) converted
    uint64_t* p_h1s = p_h1t + 1;                        // leader's copy: H1 K-slab 1 (smem) converted
    uint64_t* p_n3a = p_h1s + 1;                        // local: K-slab 0 of a tile's last chunk complete
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + Smem::TMEM_PTR);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int T = a.H + 1;
    // SS_TC_TRACE: clock stamps go to shared memory (a global store in front of a tcgen05 fence
    // would perturb the timeline) and are copied out when the kernel ends
    unsigned long long* trace_s = reinterpret_cast<unsigned long long*>(smem + Smem::TRACE);
    if (p.prof && blockIdx.x == 0)
        for (int i = tid; i < 3 * 256; i += THREADS) trace_s[i] = 0;
    unsigned long long trace_clk0 = 0, trace_ns0 = 0;
    if (p.prof && blockIdx.x == 0 && tid == 0) {
        trace_clk0 = (unsigned long long)clock64();
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(trace_ns0));
        if constexpr (PAIR) {
            // kept in shared memory (2 stamps past the events) instead of 4 registers for the whole kernel
            trace_s[3 * 256] = trace_clk0;
            trace_s[3 * 256 + 1] = trace_ns0;
        }
    }
    const int nch = p.hp / NC;          // accumulator chunks per layer
    const int nslab = p.hp / KSLAB;     // W2 K-slabs (stages) per chunk
    static_assert(KSLAB % NC == 0, "a K-slab covers whole layer-1 chunks");
    constexpr int CPS = KSLAB / NC;     // layer-1 chunks per K-slab
    const uint32_t cta_rank = cluster_ctarank();
    const bool leader = cta_rank == 0;
    const int it0 = PAIR ? 2 * p.pair_iters : 0;    // first tile iteration on the one-tile schedule

    // ---- one-time setup ----------------------------------------------------------------
    if (tid == 0) {
        for (int s = 0; s < NSTAGE; ++s) {
            mbar_init(&w2_full[s], leader ? 2 : 1);   // leader: own TMA + the peer's "landed" relay
            mbar_init(&w2_peer[s], 1);
            mbar_init(&w2_empty[s], 1);
        }
        for (int s = 0; s < ACC_SLOTS; ++s) { mbar_init(&acc_full[s], 1); mbar_init(&acc_free[s], 2 * ROW_WARPS); }
        for (int c = 0; c < HP_MAX / NC; ++c) { mbar_init(&h1_ready[c], 2 * ROW_WARPS); mbar_init(&l1_full[c], 1); }
        mbar_init(x_ready, 2 * 4);       // the four ch-0 warps of each CTA
        mbar_init(w1_full, 1);
        if constexpr (PAIR) {
            for (int s = 0; s < PAIR_STAGES; ++s) { mbar_init(&p_w2_full[s], leader ? 2 : 1); mbar_init(&p_w2_empty[s], 1); }
            for (int s = 0; s < ACC_SLOTS; ++s) { mbar_init(&p_acc_full[s], 1); mbar_init(&p_acc_free[s], 2 * ROW_WARPS); }
            mbar_init(p_x_ready, 2 * 4);
            mbar_init(p_l1a, 1);
            mbar_init(p_l1b, 1);
            mbar_init(p_scr, 2 * ROW_WARPS);
            mbar_init(p_h1t, 2 * ROW_WARPS);
            mbar_init(p_h1s, 2 * ROW_WARPS);
            mbar_init(p_n3a, 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)),
                     "n"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
    }
    for (int i = tid; i < (p.hp / 2) * (2 * DZP); i += THREADS) w3s[i] = p.w3[i];
    __syncthreads();
    if (tid == 0) {
        // this CTA's half of the layer-1 weights (resident for the whole kernel)
        mbar_expect_tx(w1_full, (uint32_t)(nch * W1_CHUNK_BYTES));
        bulk_g2s(w1s, reinterpret_cast<const unsigned char*>(p.w1_img) + (size_t)cta_rank * nch * W1_CHUNK_BYTES,
                 (uint32_t)(nch * W1_CHUNK_BYTES), w1_full);
        mbar_wait<false>(w1_full, 0);
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                  // barriers, TMEM and W1 of BOTH CTAs exist from here on
    tc_fence_after();
    const uint32_t tmem = *tmem_ptr;

    if (warp < ROW_WARPS) {
        // =============================== ROW WARPS ========================================
        const int q = warp & 3, ch = warp >> 2;
        const int row = q * 32 + lane;
        const uint32_t lane_addr = tmem + ((uint32_t)(q * 32) << 16);
        uint32_t step_it = 0;
        // state update x += (z + b3) * std_z + mean_z as one FMA per dimension: pin the two
        // constants in registers (a constant-bank miss here sits on the per-step critical path)
        float upd_s[DZ], upd_c[DZ];
#pragma unroll
        for (int j = 0; j < DZ; ++j) {
            upd_s[j] = j < a.d ? a.norm.std_z[j] : 0.f;
            upd_c[j] = j < a.d ? fmaf(__ldg(p.b3 + j), a.norm.std_z[j], a.norm.mean_z[j]) : 0.f;
            asm volatile("" : "+f"(upd_s[j]), "+f"(upd_c[j]));
        }
        if constexpr (PAIR) {
            // ========================= ROW WARPS, two-tile schedule =========================
            // Half-step h runs the layer 2 of tile x = h & 1 (step h >> 1); meanwhile these warps finish the
            // other tile y's step (its last epilogue, exchange, update, scoring, x-split) and convert its next
            // layer 1, which the MMA warp slots in between the two K-slabs of x's last chunk: chunk 0 in place
            // in y's K-slab-0 columns, chunk 1 in accumulator slot 0, chunks 2 and 3 one after the other in x's
            // K-slab-0 columns (dead once x's last chunk has read them) -> y's K-slab-1 image in smem.
            // Per tile only what the step chain carries; the sequence index is recomputed from the tile pair
            // and the Philox block of an action from its counter (no cached cursor): two tiles' state has to
            // fit next to the conversion registers under the 168-register cap of 10 warps.
            struct TileSt {
                float x[DT];
                ScoreAcc sc;
                float act[MAXIN - DZ];          // K1T = 16: every action of the shape has an input slot
            };
            TileSt ts[2];
            long long tile0 = 0;                // tile of ts[0]; ts[1] rolls tile0 + gridDim.x
            auto k_of = [&](int i) { return (tile0 + (long long)i * gridDim.x) * TM + row; };
            auto live_of = [&](int i) { return tile0 + (long long)i * gridDim.x < p.tile_end && k_of(i) < a.K_local; };
            auto qcol_of = [&](int i) {
                const long long tile = tile0 + (long long)i * gridDim.x;
                return tile < p.tile_end ? tile * 4 + q : -1ll;
            };
            auto fetch_act = [&](int i, int t) {
                ActionCursor cur;
                action_cursor_init(cur);
#pragma unroll
                for (int j = 0; j < MAXIN - DZ; ++j)
                    if (j < a.da) ts[i].act[j] = fetch_action_seq(a.act, cur, k_of(i), a.k_offset + k_of(i), t, j);
            };
            // layer-3 partial sums: only one tile has chunks in flight at a time (x's n0-n2, then its n3 first
            // thing in the next half-step); zeroed right before n0, so they hold no register during scoring
            float2 zacc[DZ];
            const long long n_qcols = 4 * ((a.K_local + TM - 1) / TM);
            unsigned char* h1s = smem + Smem::H1S;
            auto xsplit = [&](TileSt& T) {
                // as in the one-tile schedule: hi/lo split of the normalised (state, action) into A1
                float xin[MAXIN];
#pragma unroll
                for (int j = 0; j < MAXIN; ++j) xin[j] = 0.f;
#pragma unroll
                for (int j = 0; j < DZ; ++j)
                    if (j < MAXIN) xin[j] = (T.x[j] - a.norm.mean_x[j]) * a.norm.inv_std_x[j];
#pragma unroll
                for (int j = 0; j < MAXIN - DZ; ++j) xin[DZ + j] = (T.act[j] - a.norm.mean_y[j]) * a.norm.inv_std_y[j];
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
                tc_fence_before();      // this warp's last tcgen05.ld of the scratch columns precedes layer 1
                __syncwarp();
                if (lane == 0) mbar_arrive_leader(p_x_ready);
            };
            // layer-2 chunk n: relu + packed FFMA2 layer 3 into zacc
            auto epilogue = [&](int n) {
                const uint32_t slot_i = (uint32_t)(n & 1);
                mbar_wait<false>(&p_acc_full[slot_i], (uint32_t)(n >> 1) & 1);
                tc_fence_after();
                uint32_t v0[32], v1[32];
                tmem_ld32(lane_addr + COL_ACC + slot_i * NC + ch * CPT, v0);
                tmem_ld32(lane_addr + COL_ACC + slot_i * NC + ch * CPT + 32, v1);
                tmem_wait_ld();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_leader(&p_acc_free[slot_i]);
                const float* wrow = w3s + (size_t)((n * NC + ch * CPT) / 2) * (2 * DZP);
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
                        if (2 * jq + 1 < DZ) zacc[2 * jq + 1] = __ffma2_rn(hh, make_float2(w.z, w.w), zacc[2 * jq + 1]);
                    }
                }
            };
            // last chunk, exchange of the two column halves, state update (same order as the one-tile schedule)
            auto finish_step = [&](TileSt& T) {
                epilogue(3);
#pragma unroll
                for (int j = 0; j < DZ; ++j) zx[(j * TPR + ch) * TM + row] = zacc[j].x + zacc[j].y;
                asm volatile("bar.sync %0, 64;" ::"r"(2 + q) : "memory");
#pragma unroll
                for (int j = 0; j < DZ; ++j) {
                    float zz = zx[(j * TPR) * TM + row];
#pragma unroll
                    for (int o = 1; o < TPR; ++o) zz += zx[(j * TPR + o) * TM + row];
                    T.x[j] += fmaf(zz, upd_s[j], upd_c[j]);
                }
                asm volatile("bar.sync %0, 64;" ::"r"(2 + q) : "memory");   // zx is free for the other tile
            };
            // layer-1 chunk in TMEM -> relu, bf16 -> 8 K-groups of tile y's K-slab-1 image
            auto to_smem = [&](const uint32_t (&v0)[32], const uint32_t (&v1)[32], int y, int c) {
                unsigned char* img = h1s + (size_t)y * H1S_BYTES + row * 16;
#pragma unroll
                for (int g = 0; g < 8; ++g) {
                    const uint32_t(&v)[32] = g < 4 ? v0 : v1;
                    const int o = (g & 3) * 8;
                    uint4 w;
                    w.x = pack_bf16_relu(__uint_as_float(v[o + 0]), __uint_as_float(v[o + 1]));
                    w.y = pack_bf16_relu(__uint_as_float(v[o + 2]), __uint_as_float(v[o + 3]));
                    w.z = pack_bf16_relu(__uint_as_float(v[o + 4]), __uint_as_float(v[o + 5]));
                    w.w = pack_bf16_relu(__uint_as_float(v[o + 6]), __uint_as_float(v[o + 7]));
                    *reinterpret_cast<uint4*>(img + (size_t)((c - 2) * (NC / 8) + ch * (CPT / 8) + g) * (TM * 16)) = w;
                }
            };
            auto convert_l1 = [&](int y, int scr, uint32_t ev) {
                uint32_t v0[32], v1[32], pk0[16], pk1[16];
                const uint32_t ycol = (uint32_t)y * (KSLAB / 2), scol = (uint32_t)scr * (KSLAB / 2);
                mbar_wait<false>(p_l1a, ev & 1);
                tc_fence_after();
                // chunk 0: FP32 in y's K-slab-0 columns, converted in place (pair barrier: both threads loaded)
                tmem_ld32(lane_addr + ycol + ch * CPT, v0);
                tmem_ld32(lane_addr + ycol + ch * CPT + 32, v1);
                tmem_wait_ld();
                asm volatile("bar.sync %0, 64;" ::"r"(2 + q) : "memory");
#pragma unroll
                for (int c2 = 0; c2 < 16; ++c2) {
                    pk0[c2] = pack_bf16_relu(__uint_as_float(v0[2 * c2]), __uint_as_float(v0[2 * c2 + 1]));
                    pk1[c2] = pack_bf16_relu(__uint_as_float(v1[2 * c2]), __uint_as_float(v1[2 * c2 + 1]));
                }
                tmem_st16(lane_addr + ycol + ch * (CPT / 2), pk0);
                tmem_st16(lane_addr + ycol + ch * (CPT / 2) + 16, pk1);
                // chunk 1: FP32 in accumulator slot 0
                tmem_ld32(lane_addr + COL_ACC + ch * CPT, v0);
                tmem_ld32(lane_addr + COL_ACC + ch * CPT + 32, v1);
                tmem_wait_ld();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_leader(&p_acc_free[0]);
#pragma unroll
                for (int c2 = 0; c2 < 16; ++c2) {
                    pk0[c2] = pack_bf16_relu(__uint_as_float(v0[2 * c2]), __uint_as_float(v0[2 * c2 + 1]));
                    pk1[c2] = pack_bf16_relu(__uint_as_float(v1[2 * c2]), __uint_as_float(v1[2 * c2 + 1]));
                }
                tmem_st16(lane_addr + ycol + NC / 2 + ch * (CPT / 2), pk0);
                tmem_st16(lane_addr + ycol + NC / 2 + ch * (CPT / 2) + 16, pk1);
                tmem_wait_st();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_leader(p_h1t);
                // chunk 2: FP32 in x's K-slab-0 columns; once loaded they take chunk 3
                tmem_ld32(lane_addr + scol + ch * CPT, v0);
                tmem_ld32(lane_addr + scol + ch * CPT + 32, v1);
                tmem_wait_ld();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_leader(p_scr);
                to_smem(v0, v1, y, 2);
                mbar_wait<false>(p_l1b, ev & 1);
                tc_fence_after();
                tmem_ld32(lane_addr + scol + ch * CPT, v0);
                tmem_ld32(lane_addr + scol + ch * CPT + 32, v1);
                tmem_wait_ld();
                to_smem(v0, v1, y, 3);
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic -> async proxy
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_leader(p_h1s);
            };
            uint32_t ev = 0;     // layer-1 events (one per tile and step, in the MMA warp's order)
            int hs = 0;          // half-steps (SS_TC_TRACE)
            const int tb = warp == 0 ? 20 : (warp == 4 ? 40 : 64);   // other warps are not stamped
            for (int pit = 0; pit < p.pair_iters; ++pit) {
#pragma unroll
                tile0 = p.tile_begin + (long long)(2 * pit) * gridDim.x + blockIdx.x;
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    TileSt& T = ts[i];
                    load_start<ROWS, DT>(a, live_of(i), k_of(i), T.x);
                    if (ch == 1) score_init<DT>(a.plan, a.wp_index, T.x, T.sc);
#pragma unroll
                    for (int j = 0; j < MAXIN - DZ; ++j) T.act[j] = 0.f;
                    if (ch == 0 && live_of(i)) fetch_act(i, 0);
                }
                // tile 0's first layer 1 (scratch: tile 1's dead K-slab-0 columns)
                if (ch == 0) xsplit(ts[0]);
                convert_l1(0, 1, ev++);
                for (int t = 0; t < a.H; ++t) {
#pragma unroll
                    for (int x = 0; x < 2; ++x) {
                        const int y = 1 - x;
                        TileSt& X = ts[x];
                        TileSt& Y = ts[y];
                        // tile y: the step whose layer 2 ran in the previous half-step
                        PAIR_TRACE(hs, tb + 0);
                        if (x == 1 || t > 0) {
                            finish_step(Y);
                            PAIR_TRACE(hs, tb + 1);
                            if (x == 1 && t == a.H - 1 && ch == 1) {
                                score_row<DT>(a, a.H, Y.x, Y.sc, live_of(y), k_of(y), qcol_of(y), n_qcols, lane);
                                if (live_of(y) && a.scores_out) a.scores_out[k_of(y)] = Y.sc.score;
                            }
                        }
                        const int tyn = x == 0 ? t : t + 1;     // tile y's next step
                        if (tyn < a.H && ch == 0) {
                            if (live_of(y) && tyn > 0) fetch_act(y, tyn);
                            xsplit(Y);
                        }
                        PAIR_TRACE(hs, tb + 2);
                        if (ch == 1) score_row<DT>(a, t, X.x, X.sc, live_of(x), k_of(x), qcol_of(x), n_qcols, lane);
                        PAIR_TRACE(hs, tb + 3);
#pragma unroll
                        for (int j = 0; j < DZ; ++j) zacc[j] = make_float2(0.f, 0.f);
#pragma unroll 1
                        for (int n = 0; n < 3; ++n) {
                            epilogue(n);
                            PAIR_TRACE(hs, tb + 4 + n);
                        }
                        if (tyn < a.H) convert_l1(y, x, ev++);
                        PAIR_TRACE(hs, tb + 7);
                        ++hs;
                    }
                }
                finish_step(ts[1]);
                if (ch == 1) {
                    score_row<DT>(a, a.H, ts[1].x, ts[1].sc, live_of(1), k_of(1), qcol_of(1), n_qcols, lane);
                    if (live_of(1) && a.scores_out) a.scores_out[k_of(1)] = ts[1].sc.score;
                }
            }
        }
        for (int it = it0; it < p.iters; ++it) {
            const long long tile = p.tile_begin + (long long)it * gridDim.x + blockIdx.x;   // >= tile_end: padding
            const long long k_local = tile * TM + row;
            const bool live = tile < p.tile_end && k_local < a.K_local;
            const long long n_qcols = 4 * ((a.K_local + TM - 1) / TM);
            const long long qcol = tile < p.tile_end ? tile * 4 + q : -1;
            // both threads of a row keep identical copies of the state; ch 0 feeds the network
            // (critical path), ch 1 scores the trajectory in the shadow of the layer-2 MMAs
            float x[DT];
            ScoreAcc sc;
            load_start<ROWS, DT>(a, live, k_local, x);
            if (ch == 1) score_init<DT>(a.plan, a.wp_index, x, sc);
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
                const int trace_it = (warp == 0 || warp == 4) ? it : 1, trace_t = t;
                const int tb = warp == 4 ? 100 : 0;   // ch-1 warp's events live at +100
                TC_TRACE(tb + 0);
                // ---- layer-1 A operand: hi/lo split of the normalised (state, action) -------
                // slot layout (static): input j -> slots 3j (x_hi * W_hi), 3j+1 (x_hi * W_lo),
                // 3j+2 (x_lo * W_hi); bias (b_hi, b_lo) in the last two slots with a constant 1
                if (ch == 0) {
                    // state j -> input j (j < DZ), action j -> input DZ + j: all static; the
                    // statistics of unused inputs are zero, so they normalise to exactly 0
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
                    // smem image [k/8][row][8] (K-major core matrices): K1T / 8 x 16 B per row
#pragma unroll
                    for (int kc = 0; kc < K1T / 8; ++kc) {
                        uint4 v;
                        v.x = pack_bf16(slot[8 * kc], slot[8 * kc + 1]);
                        v.y = pack_bf16(slot[8 * kc + 2], slot[8 * kc + 3]);
                        v.z = pack_bf16(slot[8 * kc + 4], slot[8 * kc + 5]);
                        v.w = pack_bf16(slot[8 * kc + 6], slot[8 * kc + 7]);
                        *reinterpret_cast<uint4*>(a1s + kc * (TM * 16) + row * 16) = v;
                    }
                    TC_TRACE(60);
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic -> async proxy
                    TC_TRACE(61);
                    __syncwarp();
                    if (lane == 0) mbar_arrive_leader(x_ready);
                }
                TC_TRACE(tb + 1);
                // ---- layer-1 epilogue: relu, bf16, becomes the layer-2 A operand -------------
                // All nch layer-1 chunks are in flight at once: odd chunks accumulate in the two
                // accumulator slots, even chunks in the (currently dead) H1 columns [0,128) / [128,256)
                // and are converted in place.  The bf16 destination of chunk c, [64c, 64c+64), lies
                // inside the FP32 source of chunk c & ~1, so the two threads of a row meet at a pair
                // barrier after loading an even chunk and before anyone stores into its columns.
                static_assert(CPT == 64, "two 32-column TMEM loads per thread and chunk");
                for (int c0 = 0; c0 < nch; c0 += 2) {          // one K-slab of layer 2 per iteration
                    const uint32_t slot_i = (uint32_t)(c0 >> 1);
                    uint32_t v0[32], v1[32], pk0[16], pk1[16];
                    // even chunk: FP32 in the dead H1 columns, converted in place.  Only chunk 0 has a
                    // completion barrier of its own (an mbarrier wait costs ~100 clk even when the phase
                    // is long complete, and four of them sat on the per-step critical path); the other
                    // chunks share l1_full[1].
                    if (c0 == 0) mbar_wait<false>(&l1_full[0], step_it & 1);
                    TC_TRACE(tb + 2 + c0);
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
                    TC_TRACE(tb + 6 + c0);
                    // odd chunk: FP32 in accumulator slot c0 / 2; its loads are in flight while the even
                    // chunk's stores drain
                    if (c0 == 0) {
                        mbar_wait<false>(&l1_full[1], step_it & 1);
                        tc_fence_after();
                    }
                    TC_TRACE(tb + 3 + c0);
                    tmem_ld32(lane_addr + COL_ACC + slot_i * NC + ch * CPT, v0);
                    tmem_ld32(lane_addr + COL_ACC + slot_i * NC + ch * CPT + 32, v1);
                    // the even chunk is an A operand now: layer 2 may start on this K half right away
                    tmem_wait_st();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_leader(&h1_ready[c0]);
                    tmem_wait_ld();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_leader(&acc_free[slot_i]);
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
                    if (lane == 0) mbar_arrive_leader(&h1_ready[c0 + 1]);
                    TC_TRACE(tb + 7 + c0);
                }
                // ---- off the critical path (the tensor pipe is busy with layer 2 now) ----------
                if (ch == 1) {
                    score_row<DT>(a, t, x, sc, live, k_local, qcol, n_qcols, lane);
                } else if (ch == 0 && live && t + 1 < a.H) {
                    TC_TRACE(70);
#pragma unroll
                    for (int j = 0; j < SS_MAX_DA; ++j)
                        if (j < a.da) act[j] = fetch_action_seq(a.act, cur, k_local, a.k_offset + k_local, t + 1, j);
                    TC_TRACE(71);
                }
                TC_TRACE(tb + 19);
                // ---- layer-2 epilogue fused with layer 3 --------------------------------------
                // two hidden units per packed FFMA2: zacc[j] = (sum over even units, sum over odd units)
                float2 zacc[DZ];
#pragma unroll
                for (int j = 0; j < DZ; ++j) zacc[j] = make_float2(0.f, 0.f);
                for (int n = 0; n < nch; ++n) {
                    const uint32_t slot_i = (uint32_t)(n & 1);
                    // k-th completion of this slot: (nch + 1 - slot) / 2 layer-2 chunks per step use it
                    const uint32_t full_k = step_it * (uint32_t)((nch + 1 - (int)slot_i) >> 1) + (uint32_t)(n >> 1);
                    mbar_wait<false>(&acc_full[slot_i], full_k & 1);
                    TC_TRACE(tb + 10 + n);
                    tc_fence_after();
                    uint32_t v0[32], v1[32];
                    tmem_ld32(lane_addr + COL_ACC + slot_i * NC + ch * CPT, v0);
                    tmem_ld32(lane_addr + COL_ACC + slot_i * NC + ch * CPT + 32, v1);
                    tmem_wait_ld();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_leader(&acc_free[slot_i]);
                    const float* wrow = w3s + (size_t)((n * NC + ch * CPT) / 2) * (2 * DZP);
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
                    TC_TRACE(tb + 14 + n);
                }
                // ---- the two column halves exchange partial sums; both update the state ---------
#pragma unroll
                for (int j = 0; j < DZ; ++j) zx[(j * TPR + ch) * TM + row] = zacc[j].x + zacc[j].y;
                TC_TRACE(tb + 62);
                // only the two warps that share these rows have to meet (warp q and q + 4)
                asm volatile("bar.sync %0, 64;" ::"r"(2 + q) : "memory");
                TC_TRACE(tb + 63);
#pragma unroll
                for (int j = 0; j < DZ; ++j) {
                    // fixed order (half 0 + half 1) so both copies stay bit-identical; dimensions
                    // >= d have zero weights and zero constants: x stays 0
                    float zz = zx[(j * TPR) * TM + row];
#pragma unroll
                    for (int o = 1; o < TPR; ++o) zz += zx[(j * TPR + o) * TM + row];
                    x[j] += fmaf(zz, upd_s[j], upd_c[j]);
                }
                // (zx is rewritten only after the next step's layer-2 MMAs, which every row warp of
                // the pair has to enable through h1_ready: no second barrier needed)
                TC_TRACE(tb + 18);
            }
            if (ch == 1) {
                score_row<DT>(a, a.H, x, sc, live, k_local, qcol, n_qcols, lane);
                if (live && a.scores_out) a.scores_out[k_local] = sc.score;
            }
        }
    } else if (warp == ROW_WARPS) {
        if (leader) {
            // ============================ MMA ISSUER (leader CTA) ==============================
            // the whole warp walks the loop (warp-uniform control flow); one elected lane issues
            // every MMA of the pair (cta_group::2: rows 0-127 in this CTA's TMEM, 128-255 in the
            // peer's; B halves are read from both CTAs' shared memory at the same offset)
            // uses of accumulator slot s per step: one layer-1 chunk (c = 2s + 1, if it exists) and
            // the layer-2 chunks n with n & 1 == s; the k-th use waits for the (k-1)-th drain
            uint32_t w2_it = 0, step_it = 0;
            const uint32_t l1_use[ACC_SLOTS] = {1 < nch ? 1u : 0u, 3 < nch ? 1u : 0u};
            const uint32_t use_per_step[ACC_SLOTS] = {l1_use[0] + (uint32_t)((nch + 1) >> 1),
                                                      l1_use[1] + (uint32_t)(nch >> 1)};
            const uint32_t a1_addr = smem_u32(a1s), w1_addr = smem_u32(w1s), ring_addr = smem_u32(w2_ring);
            // layer-1 operands never change: build the descriptors once and pin them in registers
            // (the uniform-datapath arithmetic ptxas would otherwise redo per step sits on the
            // critical path between x_ready and the first layer-1 MMA)
            constexpr int NCH_MAX = HP_MAX / NC;
            uint64_t l1_a[K1T / 16], l1_b[NCH_MAX][K1T / 16];
            uint32_t l1_d[NCH_MAX], l1_bar[NCH_MAX];
#pragma unroll
            for (int ks = 0; ks < K1T / 16; ++ks) {
                l1_a[ks] = make_desc(a1_addr + ks * 2 * (TM * 16), TM);
                asm volatile("" : "+l"(l1_a[ks]));
            }
#pragma unroll
            for (int c = 0; c < NCH_MAX; ++c) {
#pragma unroll
                for (int ks = 0; ks < K1T / 16; ++ks) {
                    l1_b[c][ks] = make_desc(w1_addr + c * W1_CHUNK_BYTES + ks * 2 * (NH * 16), NH);
                    asm volatile("" : "+l"(l1_b[c][ks]));
                }
                l1_d[c] = tmem + ((c & 1) ? COL_ACC : COL_H1) + (uint32_t)(c >> 1) * NC;
                l1_bar[c] = smem_u32(&l1_full[c]);
                asm volatile("" : "+r"(l1_d[c]), "+r"(l1_bar[c]));
            }
            if constexpr (PAIR) {
                // ====================== MMA ISSUER, two-tile schedule (hp = 512) ======================
                // Static issue order of half-step h (tile x = h & 1 runs layer 2, tile y = 1 - x is one
                // half-step behind):
                //   x.n0 [slot 0] | x.n1 [slot 1] | x.n2 [slot 0] | x.n3 K-slab 0 [slot 1] |
                //   y.L1 chunks 0, 1 [y slab 0, slot 0] | (x.n3 K-slab 0 complete) y.L1 chunk 2 [x slab 0] |
                //   x.n3 K-slab 1 | (chunk 2 loaded) y.L1 chunk 3 [x slab 0]
                // Layer 2: K-slab 0 of each chunk reads A from the tile's TMEM columns, K-slab 1 from its smem
                // image (same K order as the one-tile schedule).  While x's chunks run, the row warps finish y's
                // previous step and write y's layer-1 A tile; y's layer 1 then runs between the two K-slabs of
                // x's last chunk, so its conversion hides under the 16 smem-A MMAs of that K-slab.
                // Every write into TMEM columns that an earlier MMA reads or writes waits for that MMA's
                // completion through an mbarrier: tcgen05.mma ops of one thread are ordered among themselves only
                // when they share the accumulator, and chunk 2 overwrites x's K-slab 0 (A of x.n3 K-slab 0,
                // accumulator slot 1) -- hence the commit on p_n3a.  y's slab 0 and slot 0 were last used by MMAs
                // whose completion the row warps observed before they released x.n1's slot and x.n2's slot.
                const uint32_t pring = smem_u32(smem + Smem::PRING), h1s_addr = smem_u32(smem + Smem::H1S);
                uint32_t use0 = 0, use1 = 0;             // uses of accumulator slots 0 and 1 so far
                uint32_t pw = 0, ev = 0, hs = 0;         // W2 blocks, layer-1 events, half-steps
                auto take_slot = [&](int s) {
                    uint32_t& u = s ? use1 : use0;      // s is a constant at every call: plain registers
                    mbar_wait<true>(&p_acc_free[s], (u & 1) ^ 1);
                    ++u;
                };
                auto l1_issue = [&](int c, uint32_t d) {
#pragma unroll
                    for (int ks = 0; ks < K1T / 16; ++ks) umma2_ss(d, l1_a[ks], l1_b[c][ks], IDESC, ks);
                };
                // chunks 0-2 of tile y's layer 1; scr: tile whose K-slab-0 columns take chunks 2 and 3 (after
                // its last chunk's K-slab 0 has completed when wait_scr)
                auto l1_first = [&](int y, int scr, bool wait_scr) {
                    PAIR_TRACE(hs, 18);
                    mbar_wait<true>(p_x_ready, ev & 1);
                    take_slot(0);
                    PAIR_TRACE(hs, 19);
                    tc_fence_after();
                    if (elect_one()) {
                        l1_issue(0, tmem + (uint32_t)y * (KSLAB / 2));
                        l1_issue(1, tmem + COL_ACC);
                    }
                    __syncwarp();
                    if (wait_scr) {
                        mbar_wait<true>(p_n3a, hs & 1);
                        tc_fence_after();
                    }
                    PAIR_TRACE(hs, 17);
                    if (elect_one()) {
                        l1_issue(2, tmem + (uint32_t)scr * (KSLAB / 2));
                        tc_commit_pair(p_l1a);
                    }
                    __syncwarp();
                };
                auto l1_last = [&](int scr) {
                    mbar_wait<true>(p_scr, ev & 1);
                    PAIR_TRACE(hs, 16);
                    tc_fence_after();
                    if (elect_one()) {
                        l1_issue(3, tmem + (uint32_t)scr * (KSLAB / 2));
                        tc_commit_pair(p_l1b);
                    }
                    __syncwarp();
                    ++ev;
                };
                // K-slab ksl of chunk n: two 16 KB stages of 8 MMAs each
                auto l2_slab = [&](int x, int n, int ksl) {
                    PAIR_TRACE(hs, 2 * n + ksl);
#pragma unroll
                    for (int hf = 0; hf < 2; ++hf, ++pw) {
                        const uint32_t st = pw % PAIR_STAGES;
                        if (n == 0 && hf == 0)
                            mbar_wait2(&p_w2_full[st], (pw / PAIR_STAGES) & 1, ksl ? p_h1s : p_h1t, hs & 1);
                        else
                            mbar_wait<true>(&p_w2_full[st], (pw / PAIR_STAGES) & 1);
                        tc_fence_after();
                        if (elect_one()) {
                            const uint32_t d_tmem = tmem + COL_ACC + (uint32_t)(n & 1) * NC;
                            const uint64_t b0 = make_desc(pring + st * PSTAGE_BYTES, NH);
                            if (ksl == 0) {
#pragma unroll
                                for (int ks = 0; ks < KSLAB / 32; ++ks)
                                    umma2_ts(d_tmem, tmem + (uint32_t)x * (KSLAB / 2) + (hf * KSLAB / 32 + ks) * 8,
                                             b0 + (uint64_t)((ks * 2 * (NH * 16)) >> 4), IDESC, (hf | ks) != 0);
                            } else {
                                const uint64_t a0 = make_desc(h1s_addr + (uint32_t)x * H1S_BYTES, TM);
#pragma unroll
                                for (int ks = 0; ks < KSLAB / 32; ++ks)
                                    umma2_ss(d_tmem, a0 + (uint64_t)(((hf * KSLAB / 32 + ks) * 2 * (TM * 16)) >> 4),
                                             b0 + (uint64_t)((ks * 2 * (NH * 16)) >> 4), IDESC, 1u);
                            }
                            tc_commit_pair(&p_w2_empty[st]);
                            if (ksl == 1 && hf == 1) tc_commit_pair(&p_acc_full[n & 1]);
                            if (n == 3 && ksl == 0 && hf == 1) tc_commit_pair(p_n3a);
                        }
                        __syncwarp();
                    }
                    PAIR_TRACE(hs, 8 + 2 * n + ksl);
                };
                for (int pit = 0; pit < p.pair_iters; ++pit) {
                    l1_first(0, 1, false);      // tile 1's columns: last read by MMAs the rows saw complete
                    l1_last(1);
                    for (int t = 0; t < a.H; ++t) {
#pragma unroll
                        for (int x = 0; x < 2; ++x) {
                            const bool y_next = x == 0 || t + 1 < a.H;
#pragma unroll
                            for (int n = 0; n < 3; ++n) {
                                take_slot(n & 1);
                                l2_slab(x, n, 0);
                                l2_slab(x, n, 1);
                            }
                            take_slot(1);
                            l2_slab(x, 3, 0);
                            if (y_next) l1_first(1 - x, x, true);
                            l2_slab(x, 3, 1);
                            if (y_next) l1_last(x);
                            ++hs;
                        }
                    }
                }
            }
            for (int it = it0; it < p.iters; ++it) {
                for (int t = 0; t < a.H; ++t, ++step_it) {
                    const int trace_it = it, trace_t = t;
                    // layer 1: chunk c = A1 [256 x K1T] * W1img[c] [128 x K1T]^T; odd chunks go to the
                    // accumulator slots (once the previous step's layer-2 epilogue drained them --
                    // long before x_ready, so these ~90-cycle waits are taken off the critical path),
                    // even chunks to the dead H1 columns -- all issued back to back
                    // (all of these completed long before x_ready: polled together, off the critical path;
                    // the first W2 stage of the step is taken here as well)
                    if (l1_use[1])
                        mbar_wait2(&acc_free[0], ((step_it * use_per_step[0]) & 1) ^ 1, &acc_free[1],
                                   ((step_it * use_per_step[1]) & 1) ^ 1);
                    else if (l1_use[0])
                        mbar_wait<true>(&acc_free[0], ((step_it * use_per_step[0]) & 1) ^ 1);
                    mbar_wait<true>(&w2_full[w2_it % NSTAGE], (w2_it / NSTAGE) & 1);
                    mbar_wait<true>(x_ready, step_it & 1);
                    TC_TRACE(20);
                    tc_fence_after();
                    if (elect_one()) {
#pragma unroll
                        for (int c = 0; c < NCH_MAX; ++c)
                            if (c < nch) {
#pragma unroll
                                for (int ks = 0; ks < K1T / 16; ++ks) umma2_ss(l1_d[c], l1_a[ks], l1_b[c][ks], IDESC, ks);
                                // chunk 0 completes on its own barrier (the row warps start converting
                                // it at once), all the others on l1_full[1]
                                if (c == 0) tc_commit_pair_addr(l1_bar[0]);
                                else if (c == nch - 1) tc_commit_pair_addr(l1_bar[1]);
                            }
                    }
                    __syncwarp();
                    TC_TRACE(21);
                    // layer 2: acc chunk n = H1 [256 x HP] * W2img[n] [128 x HP]^T, K streamed in slabs
                    for (int n = 0; n < nch; ++n) {
                        const uint32_t slot_i = (uint32_t)(n & 1);
                        const uint32_t free_k = slot_i ? step_it * use_per_step[1] + l1_use[1] + (uint32_t)(n >> 1)
                                                       : step_it * use_per_step[0] + l1_use[0] + (uint32_t)(n >> 1);
                        // accumulator slot drained by its previous user.  For n == 0 that user is layer-1
                        // chunk 1: every row warp arrives here AFTER it arrived on h1_ready[0] (program
                        // order, both release), so this one wait also covers "H1 chunk 0 is converted".
                        // For n >= 1 the wait is polled together with the first W2 stage of the chunk.
                        if (n == 0 || nslab < 1) mbar_wait<true>(&acc_free[slot_i], (free_k & 1) ^ 1);
                        else mbar_wait2(&acc_free[slot_i], (free_k & 1) ^ 1, &w2_full[w2_it % NSTAGE], (w2_it / NSTAGE) & 1);
                        TC_TRACE(41 + n);
                        for (int ksl = 0; ksl < nslab; ++ksl, ++w2_it) {
                            const uint32_t st = w2_it % NSTAGE;
                            const uint32_t d_tmem = tmem + COL_ACC + slot_i * NC;
                            const uint32_t a_tmem = tmem + COL_H1 + ksl * (KSLAB / 2);
                            const uint64_t b0 = make_desc(ring_addr + st * STAGE_BYTES, NH);
                            if (n == 0) {
                                // first chunk of the step: the A operand is still being converted -- issue
                                // each 128-wide K half as soon as ITS layer-1 chunk is ready.  The W2 stage of
                                // K-slab 0 was taken before x_ready; later slabs poll it together with h1_ready.
                                static_assert(CPS == 2, "two layer-1 chunks per K-slab");
                                if (ksl > 0)
                                    mbar_wait2(&w2_full[st], (w2_it / NSTAGE) & 1, &h1_ready[ksl * CPS], step_it & 1);
                                else if (l1_use[0] == 0)
                                    mbar_wait<true>(&h1_ready[0], step_it & 1);     // (no layer-1 chunk in slot 0)
                                TC_TRACE(45 + 2 * ksl);
                                tc_fence_after();
                                if (elect_one()) {
#pragma unroll
                                    for (int ks = 0; ks < KSLAB / 32; ++ks)
                                        umma2_ts(d_tmem, a_tmem + ks * 8, b0 + (uint64_t)((ks * 2 * (NH * 16)) >> 4), IDESC,
                                                 (ksl | ks) != 0);
                                }
                                __syncwarp();
                                mbar_wait<true>(&h1_ready[ksl * CPS + 1], step_it & 1);
                                TC_TRACE(46 + 2 * ksl);
                                tc_fence_after();
                                if (elect_one()) {
#pragma unroll
                                    for (int ks = KSLAB / 32; ks < KSLAB / 16; ++ks)
                                        umma2_ts(d_tmem, a_tmem + ks * 8, b0 + (uint64_t)((ks * 2 * (NH * 16)) >> 4), IDESC, 1u);
                                    tc_commit_pair(&w2_empty[st]);
                                    if (ksl == nslab - 1) tc_commit_pair(&acc_full[slot_i]);
                                }
                            } else {
                                if (ksl > 0) mbar_wait<true>(&w2_full[st], (w2_it / NSTAGE) & 1);    // both halves have landed
                                tc_fence_after();
                                if (elect_one()) {
#pragma unroll
                                    for (int ks = 0; ks < KSLAB / 16; ++ks)
                                        umma2_ts(d_tmem, a_tmem + ks * 8, b0 + (uint64_t)((ks * 2 * (NH * 16)) >> 4), IDESC,
                                                 (ksl | ks) != 0);
                                    tc_commit_pair(&w2_empty[st]);
                                    if (ksl == nslab - 1) tc_commit_pair(&acc_full[slot_i]);
                                }
                            }
                            __syncwarp();
                            TC_TRACE(25 + n * 4 + ksl);
                        }
                    }
                }
            }
        } else {
            // ============================ STAGE RELAY (peer CTA) ===============================
            // tell the leader's MMA warp when this CTA's half of a W2 stage has landed
            if (lane == 0) {
                if constexpr (PAIR) {
                    const long long ptotal = (long long)p.pair_iters * 2 * a.H * nch * nslab * 2;
                    for (long long i = 0; i < ptotal; ++i) {
                        const uint32_t st = (uint32_t)(i % PAIR_STAGES);
                        mbar_wait<false>(&p_w2_full[st], (uint32_t)(i / PAIR_STAGES) & 1);
                        mbar_arrive_leader(&p_w2_full[st]);
                    }
                }
                uint32_t w2_it = 0;
                const long long total = (long long)(p.iters - it0) * a.H * nch * nslab;
                for (long long i = 0; i < total; ++i, ++w2_it) {
                    const uint32_t st = w2_it % NSTAGE;
                    mbar_wait<false>(&w2_full[st], (w2_it / NSTAGE) & 1);
                    mbar_arrive_leader(&w2_full[st]);
                }
            }
        }
    } else {
        // =============================== TMA PRODUCER =====================================
        if (lane == 0) {
            const int blocks = nch * nslab;
            if constexpr (PAIR) {
                // the two-tile stream: one W2 pass per half-step in the MMA warp's issue order, each 32 KB block
                // as two 16 KB stages (K 0-127, K 128-255 of the slab: contiguous in the K-major image)
                const long long ptotal = (long long)p.pair_iters * 2 * a.H * blocks * 2;
                for (long long i = 0; i < ptotal; ++i) {
                    const uint32_t st = (uint32_t)(i % PAIR_STAGES);
                    const long long blk = (i >> 1) % blocks;
                    mbar_wait<false>(&p_w2_empty[st], ((uint32_t)(i / PAIR_STAGES) & 1) ^ 1);
                    mbar_expect_tx(&p_w2_full[st], PSTAGE_BYTES);
                    bulk_g2s(smem + Smem::PRING + (size_t)st * PSTAGE_BYTES,
                             reinterpret_cast<const unsigned char*>(p.w2_img) +
                                 ((size_t)blk * CLUSTER + cta_rank) * STAGE_BYTES + (size_t)(i & 1) * PSTAGE_BYTES,
                             PSTAGE_BYTES, &p_w2_full[st]);
                }
                // the one-tile ring overwrites the H1 images: wait for the last two-tile MMA (in-order completion)
                for (long long i = ptotal - PAIR_STAGES; i < ptotal; ++i)
                    if (i >= 0) mbar_wait<false>(&p_w2_empty[i % PAIR_STAGES], (uint32_t)(i / PAIR_STAGES) & 1);
            }
            uint32_t w2_it = 0;
            for (int it = it0; it < p.iters; ++it)
                for (int t = 0; t < a.H; ++t)
                    for (int blk = 0; blk < blocks; ++blk, ++w2_it) {
                        const uint32_t st = w2_it % NSTAGE;
                        // drained by the pair's MMAs (the commit is multicast to both CTAs)
                        mbar_wait<false>(&w2_empty[st], ((w2_it / NSTAGE) & 1) ^ 1);
                        mbar_expect_tx(&w2_full[st], STAGE_BYTES);
                        bulk_g2s(w2_ring + (size_t)st * STAGE_BYTES,
                                 reinterpret_cast<const unsigned char*>(p.w2_img) +
                                     ((size_t)blk * CLUSTER + cta_rank) * STAGE_BYTES,
                                 STAGE_BYTES, &w2_full[st]);
                    }
        }
    }
    // ---- teardown ---------------------------------------------------------------------------
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                  // no CTA leaves while its peer may still read / signal it
    tc_fence_after();
    if (p.prof && blockIdx.x == 0) {
        for (int i = tid; i < 3 * 256; i += THREADS) p.prof[i] = trace_s[i];
        if (tid == 0) {
            // SM clock actually delivered over the kernel: cycles / globaltimer nanoseconds
            unsigned long long ns1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns1));
            if constexpr (PAIR) {
                trace_clk0 = trace_s[3 * 256];
                trace_ns0 = trace_s[3 * 256 + 1];
            }
            p.prof[3 * 256] = (unsigned long long)clock64() - trace_clk0;
            p.prof[3 * 256 + 1] = ns1 - trace_ns0;
        }
    }
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(TMEM_COLS));
}

// ---- host side ---------------------------------------------------------------------------
static uint16_t bf16_bits(float f) {
    uint32_t u;
    std::memcpy(&u, &f, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);   // NaN
    u += 0x7fffu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}
static float bf16_val(uint16_t b) {
    uint32_t u = (uint32_t)b << 16;
    float f;
    std::memcpy(&f, &u, 4);
    return f;
}

}  // namespace tc

bool mpc_tc_shape_supported(const ss_ctx* c) {
    // two hidden layers, hidden width + the two constant-one bias units within 512, small I/O dims
    return c->L == 2 && c->h >= 64 && c->h + 2 <= tc::HP_MAX && c->d <= 8 && tc::dz_of(c->d) + c->da <= tc::MAX_DIN;
}

int mpc_tc_prepare(ss_ctx* c) {
    using namespace tc;
    const int h = c->h, d = c->d, din = c->d + c->da;
    const int k1 = k1_slots(d, c->da), dz = dz_of(d);
    const int W1_CHUNK_BYTES = NH * k1 * 2;
    const int hp = (h + 2 + KSLAB - 1) / KSLAB * KSLAB;
    const int nch = hp / NC, nslab = hp / KSLAB;
    const std::vector<double>&W1 = c->hw[0], &W2 = c->hw[1], &W3 = c->hw[2];
    const std::vector<double>&B1 = c->hb[0], &B2 = c->hb[1];
    // Every B tile is split by output unit over the CTA pair: units [128 c + 64 r, +64) of chunk c
    // live in CTA r.  Images are [k/8][64 units][8 k] (K-major, no-swizzle core matrices).
    // layer-1 image: K slots (3j, 3j+1, 3j+2) = (W_hi, W_lo, W_hi) of input j; (b_hi, b_lo) in the
    // last two of the k1 slots
    std::vector<uint16_t> w1((size_t)CLUSTER * nch * (W1_CHUNK_BYTES / 2), 0);
    auto w1_at = [&](int slot, int u) -> uint16_t& {
        const int cidx = u / NC, r = (u % NC) / NH, nn = u % NH;
        return w1[((size_t)r * nch + cidx) * (W1_CHUNK_BYTES / 2) + (slot / 8) * (NH * 8) + nn * 8 + (slot % 8)];
    };
    for (int u = 0; u < h; ++u) {
        for (int j = 0; j < din; ++j) {
            const float w = (float)W1[(size_t)j * h + u];
            const uint16_t hi = bf16_bits(w), lo = bf16_bits(w - bf16_val(hi));
            const int in = j < d ? j : dz + (j - d);      // input slot of network input j
            w1_at(3 * in, u) = hi;
            w1_at(3 * in + 1, u) = lo;
            w1_at(3 * in + 2, u) = hi;
        }
        const float b = (float)B1[u];
        const uint16_t hi = bf16_bits(b), lo = bf16_bits(b - bf16_val(hi));
        w1_at(k1 - 2, u) = hi;
        w1_at(k1 - 1, u) = lo;
    }
    // constant-one hidden units h and h+1 (carry the layer-2 bias through the GEMM)
    w1_at(k1 - 2, h) = bf16_bits(1.f);
    w1_at(k1 - 2, h + 1) = bf16_bits(1.f);
    // layer-2 image: blocks (n, kslab, cta) of [16 k-chunks][64 units][8 k]
    std::vector<uint16_t> w2((size_t)nch * nslab * CLUSTER * (STAGE_BYTES / 2), 0);
    auto w2_at = [&](int k, int u) -> uint16_t& {
        const int n = u / NC, r = (u % NC) / NH, nn = u % NH, ksl = k / KSLAB, kk = k % KSLAB;
        return w2[(((size_t)n * nslab + ksl) * CLUSTER + r) * (STAGE_BYTES / 2) + (kk / 8) * (NH * 8) + nn * 8 +
                  (kk % 8)];
    };
    for (int u = 0; u < h; ++u) {
        for (int k = 0; k < h; ++k) w2_at(k, u) = bf16_bits((float)W2[(size_t)k * h + u]);
        const float b = (float)B2[u];
        const uint16_t hi = bf16_bits(b), lo = bf16_bits(b - bf16_val(hi));
        w2_at(h, u) = hi;
        w2_at(h + 1, u) = lo;
    }
    // layer 3 (FP32, in shared memory): [hp / 2 (unit pairs)][dzp outputs][2 units] for FFMA2
    const int dzp = w3_pair_floats(dz) / 2;
    std::vector<float> w3((size_t)hp * dzp, 0.f);
    for (int u = 0; u < h; ++u)
        for (int j = 0; j < d; ++j) w3[((size_t)(u / 2) * dzp + j) * 2 + (u & 1)] = (float)W3[(size_t)u * d + j];
    SS_CUDA_CHECK(c, c->tc_w1.ensure(w1.size() * 2));
    SS_CUDA_CHECK(c, c->tc_w2.ensure(w2.size() * 2));
    SS_CUDA_CHECK(c, c->tc_w3.ensure(w3.size() * 4));
    float b3[SS_MAX_D] = {};
    for (int j = 0; j < d; ++j) b3[j] = (float)c->hb[2][j];
    SS_CUDA_CHECK(c, c->tc_b3.ensure(SS_MAX_D * 4));
    SS_CUDA_CHECK(c, cudaMemcpyAsync(c->tc_b3.p, b3, SS_MAX_D * 4, cudaMemcpyHostToDevice, c->stream));
    SS_CUDA_CHECK(c, cudaMemcpyAsync(c->tc_w1.p, w1.data(), w1.size() * 2, cudaMemcpyHostToDevice, c->stream));
    SS_CUDA_CHECK(c, cudaMemcpyAsync(c->tc_w2.p, w2.data(), w2.size() * 2, cudaMemcpyHostToDevice, c->stream));
    SS_CUDA_CHECK(c, cudaMemcpyAsync(c->tc_w3.p, w3.data(), w3.size() * 4, cudaMemcpyHostToDevice, c->stream));
    SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
    c->tc_hp = hp;
    c->tc_dz = dz;
    c->tc_k1 = k1;
    c->tc_ready = true;
    return SS_OK;
}

int mpc_tc_tile_rows() { return tc::TM; }

// geometry of the operand images for ss_dyn_commit (dyn_train.cu), which re-packs them on the device
void mpc_tc_geometry(const ss_ctx* c, int* k1, int* dz, int* hp, int* NC_, int* NH_, int* KSLAB_, int* CLUSTER_,
                     int* dzp) {
    *k1 = c->tc_k1;
    *dz = c->tc_dz;
    *hp = c->tc_hp;
    *NC_ = tc::NC; *NH_ = tc::NH; *KSLAB_ = tc::KSLAB; *CLUSTER_ = tc::CLUSTER;
    *dzp = tc::w3_pair_floats(c->tc_dz) / 2;
}

int mpc_tc_grid(const ss_ctx* c, long long tiles) {
    // a multiple of the pair size; at most one CTA per SM (TMEM: 512 columns per CTA)
    const long long up = (tiles + tc::CLUSTER - 1) / tc::CLUSTER * tc::CLUSTER;
    const long long cap = c->sm_count / tc::CLUSTER * tc::CLUSTER;
    return (int)(up < cap ? up : cap);
}

int mpc_tc_launch(ss_ctx* c, const RolloutArgs& a, int* grid_blocks_out, long long tile_begin, long long tile_count) {
    using namespace tc;
    if (!c->tc_ready) SS_FAIL(c, SS_EUNSUPPORTED, "mpc: tcgen05 kernel not prepared for this model");
    Params p;
    std::memset(&p, 0, sizeof(p));
    p.w1_img = c->tc_w1.as<__nv_bfloat16>();
    p.w2_img = c->tc_w2.as<__nv_bfloat16>();
    p.w3 = c->tc_w3.as<float>();
    p.b3 = c->tc_b3.as<float>();
    p.hp = c->tc_hp;
    p.din = c->d + c->da;
    const long long all_tiles = (a.K_local + TM - 1) / TM;
    if (tile_count < 0) tile_count = all_tiles - tile_begin;
    if (tile_begin < 0 || tile_count < 1 || tile_begin + tile_count > all_tiles)
        SS_FAIL(c, SS_EINVAL, "mpc: tile range outside the batch");
    p.tile_begin = tile_begin;
    p.tile_end = tile_begin + tile_count;
    p.prof = nullptr;
    if (getenv("SS_TC_TRACE")) {
        SS_CUDA_CHECK(c, c->tc_misc.ensure((3 * 256 + 2) * 8));
        SS_CUDA_CHECK(c, cudaMemsetAsync(c->tc_misc.p, 0, (3 * 256 + 2) * 8, c->stream));
        p.prof = c->tc_misc.as<unsigned long long>();
    }
    const int grid = mpc_tc_grid(c, tile_count);
    if (grid_blocks_out) *grid_blocks_out = grid;
    p.iters = (int)((tile_count + grid - 1) / grid);
    // two-tile schedule: tiles go to a CTA two at a time, an odd last one runs on the one-tile schedule.
    // SS_TC_PAIR=0 forces the one-tile schedule (tests compare the two).
    const char* pair_env = getenv("SS_TC_PAIR");
    const bool pair = pair_layout_fits(c->tc_dz, c->tc_k1) && c->tc_hp == HP_MAX && p.iters >= 2 &&
                      !(pair_env && std::atoi(pair_env) == 0);
    p.pair_iters = pair ? p.iters / 2 : 0;
    c->run.tc_schedule = pair ? 1 : 0;
    const size_t trace_bytes = p.prof ? 3 * 256 * 8 : 0;
    cudaLaunchConfig_t cfg;
    std::memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(THREADS);
    cfg.stream = c->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CLUSTER;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e;
    // the instantiation whose input slots and W3 stride are the ones the images were packed with
    const int dz = c->tc_dz, k1 = c->tc_k1;
#define TC_LAUNCH(DT_, DZ_, K1_)                                                                              \
    do {                                                                                                      \
        cfg.dynamicSmemBytes = SmemT<DZ_>::END + 128 + trace_bytes;                                          \
        auto kern = a.state0_rows ? mpc_rollout_tc_kernel<DT_, DZ_, K1_, true>                                \
                                  : mpc_rollout_tc_kernel<DT_, DZ_, K1_, false>;                               \
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cfg.dynamicSmemBytes); \
        if (e == cudaSuccess) e = cudaLaunchKernelEx(&cfg, kern, a, p);                                       \
    } while (0)
#define TC_LAUNCH_PAIR(DT_, DZ_, K1_)                                                                         \
    do {                                                                                                      \
        cfg.dynamicSmemBytes = SmemT<DZ_, true>::END + 128 + (trace_bytes ? trace_bytes + 16 : 0);            \
        auto kern = a.state0_rows ? mpc_rollout_tc_kernel<DT_, DZ_, K1_, true, true>                          \
                                  : mpc_rollout_tc_kernel<DT_, DZ_, K1_, false, true>;                         \
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cfg.dynamicSmemBytes); \
        if (e == cudaSuccess) e = cudaLaunchKernelEx(&cfg, kern, a, p);                                       \
    } while (0)
    if (pair && dz == 2) TC_LAUNCH_PAIR(4, 2, 16);
    else if (pair && dz == 3) TC_LAUNCH_PAIR(4, 3, 16);
    else if (dz == 2 && k1 == 16) TC_LAUNCH(4, 2, 16);     // e.g. MountainCar (d = 2, da = 1)
    else if (dz == 2 && k1 == 32) TC_LAUNCH(4, 2, 32);     // d <= 2, da = 3 .. 8
    else if (dz == 3 && k1 == 16) TC_LAUNCH(4, 3, 16);     // e.g. Pendulum (d = 3, da = 1)
    else if (dz == 3 && k1 == 32) TC_LAUNCH(4, 3, 32);     // d = 3, da = 2 .. 7
    else if (dz == 4 && k1 == 32) TC_LAUNCH(4, 4, 32);
    else if (dz == 8 && k1 == 32) TC_LAUNCH(8, 8, 32);
    else SS_FAIL(c, SS_EUNSUPPORTED, "mpc: no tcgen05 kernel for this layer-1 layout");
#undef TC_LAUNCH
#undef TC_LAUNCH_PAIR
    if (e == cudaSuccess) e = cudaGetLastError();
    c->launches++;
    SS_CUDA_CHECK(c, e);
    if (p.prof && pair) {
        std::vector<unsigned long long> h(3 * 256 + 2);
        SS_CUDA_CHECK(c, cudaMemcpyAsync(h.data(), p.prof, h.size() * 8, cudaMemcpyDeviceToHost, c->stream));
        SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
        fprintf(stderr, "[trace] block 0: %llu clk in %llu ns = %.0f MHz delivered SM clock (two-tile schedule)\n",
                h[3 * 256], h[3 * 256 + 1], h[3 * 256 + 1] ? 1e3 * (double)h[3 * 256] / (double)h[3 * 256 + 1] : 0.0);
        const unsigned long long t0 = h[0];
        for (int hs = 0; hs < 6; ++hs) {
            fprintf(stderr, "[trace half-step %d: tile %d layer 2, tile %d finishing] mma", 20 + hs, hs & 1, 1 - (hs & 1));
            for (int e = 0; e < 20; ++e) fprintf(stderr, " %d:%lld", e, h[hs * 64 + e] ? (long long)(h[hs * 64 + e] - t0) : -1);
            for (int w = 20; w <= 40; w += 20) {
                fprintf(stderr, " | ch%d", w / 20 - 1);
                for (int e = 0; e < 8; ++e)
                    fprintf(stderr, " %d:%lld", e, h[hs * 64 + w + e] ? (long long)(h[hs * 64 + w + e] - t0) : -1);
            }
            fprintf(stderr, "\n");
        }
    } else if (p.prof) {
        std::vector<unsigned long long> h(3 * 256 + 2);
        SS_CUDA_CHECK(c, cudaMemcpyAsync(h.data(), p.prof, h.size() * 8, cudaMemcpyDeviceToHost, c->stream));
        SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
        fprintf(stderr, "[trace] block 0: %llu clk in %llu ns = %.0f MHz delivered SM clock\n", h[3 * 256], h[3 * 256 + 1],
                h[3 * 256 + 1] ? 1e3 * (double)h[3 * 256] / (double)h[3 * 256 + 1] : 0.0);
        for (int st2 = 0; st2 < 3; ++st2) {
            const unsigned long long* ev = &h[st2 * 256];
            const unsigned long long t0 = ev[0];
            fprintf(stderr, "[trace step %d] row: xsplit_done %llu | L1 full", 10 + st2, ev[1] - t0);
            for (int c2 = 0; c2 < 4; ++c2) fprintf(stderr, " %llu", ev[2 + c2] - t0);
            fprintf(stderr, " | L1 epi_done");
            for (int c2 = 0; c2 < 4; ++c2) fprintf(stderr, " %llu", ev[6 + c2] - t0);
            fprintf(stderr, " | L2 full");
            for (int c2 = 0; c2 < 4; ++c2) fprintf(stderr, " %llu", ev[10 + c2] - t0);
            fprintf(stderr, " | L2 epi_done");
            for (int c2 = 0; c2 < 4; ++c2) fprintf(stderr, " %llu", ev[14 + c2] - t0);
            fprintf(stderr, " | step_end %llu\n", ev[18] - t0);
            fprintf(stderr, "[trace step %d] detail: slots_stored %llu fence_done %llu | zx_stored %llu (ch1 %llu) bar_done %llu (ch1 %llu) | prefetch %llu .. %llu\n",
                    10 + st2, ev[60] - t0, ev[61] - t0, ev[62] - t0, ev[162] - t0, ev[63] - t0, ev[163] - t0, ev[70] - t0, ev[71] - t0);
            fprintf(stderr, "[trace step %d] mma: x_ready %llu | L1 issued", 10 + st2, ev[20] - t0);
            for (int c2 = 0; c2 < 4; ++c2) fprintf(stderr, " %llu", ev[21 + c2] - t0);
            fprintf(stderr, " | L2 slab issued");
            for (int c2 = 0; c2 < 16; ++c2) fprintf(stderr, " %llu", ev[25 + c2] - t0);
            fprintf(stderr, " | acc_free seen");
            for (int c2 = 0; c2 < 4; ++c2) fprintf(stderr, " %llu", ev[41 + c2] - t0);
            fprintf(stderr, " | n=0: h1_ready chunk0 %llu chunk1 %llu chunk2 %llu chunk3 %llu", ev[45] - t0, ev[46] - t0,
                    ev[47] - t0, ev[48] - t0);
            fprintf(stderr, "\n[trace step %d] ch1: L1 epi_done %llu | score_done %llu | L2 full", 10 + st2, ev[109] - t0, ev[119] - t0);
            for (int c2 = 0; c2 < 4; ++c2) fprintf(stderr, " %llu", ev[110 + c2] - t0);
            fprintf(stderr, " | L2 epi_done");
            for (int c2 = 0; c2 < 4; ++c2) fprintf(stderr, " %llu", ev[114 + c2] - t0);
            fprintf(stderr, " | ch0 prefetch_done %llu\n", ev[19] - t0);
        }
    }
    return SS_OK;
}
