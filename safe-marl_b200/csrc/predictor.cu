// predictor.cu -- safety-signal voltage predictor + safety penalty on tcgen05 tensor cores,
// writing straight into a device-resident replay ring (BASELINE config 4).
//
//   fp_predictor_load / fp_predict   replace `model.predict` of the reference's regressor
//       (safety_signal/train_safety_signal_model.py:33-46,73: MinMax-scaled X[66] -> 33 linear
//        outputs; interleaved input layout [P1,Q1,...,P33,Q33], data_generation.py:48-50) and the
//       slack penalty of the safety layer at fixed actions
//       (madrl/models/safemaddpg.py:205-229,264-277: 1000 * sum(max(0, v_min - V) + max(0, V - v_max)))
//   fp_predictor_load_mlp / fp_predict_mlp   the same with the regressor swapped for scikit-learn's MLPRegressor
//       (k_predict_mlp, below k_predict; both end in predict_epilogue)
//   fp_replay_*                      replace TransReplayBuffer (utils/replay_buffer.py:3-30)
//
// Kernel k_predict: one persistent CTA per SM (17 warps), 128-env tiles, WARP-SPECIALISED so that the
// phases of consecutive tiles overlap.  The op is HBM-bound by shape (K = 66, N = 33: ~11 flop/B); the
// job of the kernel is to keep five tiles of X in flight per SM while everything else hides underneath,
// and to keep shared-memory traffic (the second bound: 128 B/clk/SM) to the X tile and the Vhat tile.
//   TMA/MMA warp 16 (one elected thread)
//     1. TMA: `cp.async.bulk` brings a tile's X rows (128 x 66 fp32 = 33 792 contiguous bytes) into one
//        of FIVE staging buffers, completion on an mbarrier; a buffer is refilled (five tiles ahead) as
//        soon as every producer has read it.
//     3. tcgen05.mma (kind::tf32, M=128, N=48, K=8 per instruction; 9 k-steps x 3 products
//        hi*hi + lo*hi + hi*lo) with the A OPERAND IN TMEM and the weights (hi and lo parts, UMMA K-major
//        no-swizzle layout: [k-chunk][n][4 floats], SBO = 128 B, LBO = 48 * 16 B) in shared memory for the
//        lifetime of the CTA; fp32 accumulation in one of TWO TMEM accumulators; completion via
//        tcgen05.commit -> mbarrier.
//   producer warps 0-7 (two threads per env row of the tile: K halves)
//     2. 3xTF32 split: x = hi + lo with hi exactly representable in TF32 (low 13 mantissa bits cleared)
//        and lo = x - hi (exact).  A thread owns a row, and a TMEM lane IS a row: `tcgen05.st.32x32b.x4`
//        writes hi and lo straight into one of TWO A buffers in TMEM (lane = env row, column = k;
//        144 columns per buffer), so A never touches shared memory (it would cost 70 KB of stores and
//        110 KB of operand reads per tile there) and the split of tile i+1 overlaps the MMAs of tile i.
//   epilogue warps 8-15 (two threads per env row: column halves; TMEM lane quarter = warp % 4)
//     4. tcgen05.ld (32x32b.x16 + .x1) hands every thread its 17 / 16 accumulators of its env and frees
//        the accumulator for the tile after next; add the bias, evaluate the slack penalty (fp64, only
//        for rows that leave the limits), stage Vhat in shared memory; ONE bulk store per destination
//        (TMA engine) writes the tile into the replay ring at (pos + env) mod capacity and/or a dense
//        output (a wrapping or unaligned segment falls back to a coalesced store loop).
// TMEM map (512 columns): accumulators at 0 and 64, A buffers at 128 and 272 (hi 72 | lo 72 columns).
// The weights arrive by one bulk copy that overlaps the first X tiles (own mbarrier).  The groups meet
// only through mbarriers (full[5], a_ready[2], mma_done[2], tmem_free[2]); the epilogue synchronises
// internally with a named barrier; every wait is bounded (trap, never a hung GPU).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "api_handle.cuh"
#include "flex_handle.cuh"
#include "sm100_ptx.cuh"

namespace {

constexpr int N_IN = 66, N_OUT = 33;
constexpr uint32_t B_BYTES = PRED_KC * PRED_N * 16;          // 13 824
constexpr uint32_t STAGE_BYTES = PRED_M * N_IN * 4;          // 33 792
constexpr uint32_t OFF_BHI = 0, OFF_BLO = OFF_BHI + B_BYTES;
constexpr int N_STAGES = 5;                                  // X tiles in flight per SM (5 x 33 KB covers the HBM latency)
constexpr uint32_t OFF_STAGE = OFF_BLO + B_BYTES;
constexpr uint32_t OFF_OUT = OFF_STAGE + N_STAGES * STAGE_BYTES;   // [128][33] fp32
constexpr uint32_t OFF_BIAS = OFF_OUT + PRED_M * N_OUT * 4;
constexpr uint32_t OFF_BAR = OFF_BIAS + PRED_N * 4;          // full[5], mma_done[2], tmem_free[2], weights, a_ready[2]
constexpr uint32_t OFF_PEN = OFF_BAR + 12 * 8;                // [2][128] fp64 penalty partials (column halves)
constexpr uint32_t OFF_TMEM = OFF_PEN + 2 * PRED_M * 8;
constexpr uint32_t SMEM_BYTES = OFF_TMEM + 16;
constexpr uint32_t ACC_COLS = 64;                            // one accumulator (48 columns used)
constexpr uint32_t A_COL0 = 2 * ACC_COLS;                    // A operand in TMEM: [2 buffers][hi 72 | lo 72] columns, lane = env row
constexpr uint32_t A_COLS = 2 * PRED_K;
constexpr uint32_t TMEM_COLS = 512;                          // 2 accumulators + 2 A buffers = 416 columns -> the whole TMEM (one CTA per SM)
static_assert(SMEM_BYTES <= 227 * 1024, "predictor tile buffers exceed the shared memory of one SM");

struct PredParams {
    const float* X; int64_t n;
    const float* B; const float* bias;
    float* vhat; double* penalty;                            // dense outputs (may be null)
    float* ring_vhat; float* ring_pen; int64_t ring_cap, ring_pos;   // replay sink (may be null)
    double v_min, v_max, w;
    float lo_f, hi_f;                                        // smallest float >= v_min, largest float <= v_max
};

constexpr uint32_t IDESC = umma_idesc_tf32(PRED_M, PRED_N);

constexpr int PROD_THREADS = 2 * PRED_M;     // warps 0-7: TMA + split (two threads per row) + MMA issue (warp 0)
constexpr int EPI_THREADS = 2 * PRED_M;      // warps 8-15: epilogue (two threads per row: column halves)
constexpr int MMA_WARP = (PROD_THREADS + EPI_THREADS) / 32;   // warp 16: TMA + tcgen05.mma issue
constexpr int PRED_THREADS = PROD_THREADS + EPI_THREADS + 32;

// 3xTF32 split x = hi + lo.  Truncating (k_predict): hi = x with the low 13 mantissa bits cleared, lo = x - hi (exact,
// |lo| < 2^-10 |x|; the tensor core truncates lo to TF32 in turn).  Nearest (k_predict_mlp): hi and lo rounded to the
// nearest TF32 value, |lo| <= 2^-11 |x| and lo's own rounding <= 2^-22 |x|, a quarter of the truncating split's error
// per product, which the MLP's hidden layers, with their cancellations, need for 1e-6 p.u.
template <bool NEAREST>
__device__ __forceinline__ void tf32_split(float x, float& hi, float& lo) {
    if (NEAREST) { hi = tf32_rna(x); lo = tf32_rna(x - hi); }
    else { hi = __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); lo = x - hi; }
}

// A thread's half of one X row (K half `half`: 4-k chunks 0..8 or 9..17) as the 3xTF32 split x = hi + lo, stored at the
// thread's TMEM lane: hi at column t_hi + k, lo at t_lo + k, k = 66..71 zero.  Shared by k_predict (truncating split)
// and the first layer of k_predict_mlp (nearest).
template <bool NEAREST>
__device__ __forceinline__ void split_x_to_tmem(const float* xrow, int half, uint32_t t_hi, uint32_t t_lo) {
    const float2* src = reinterpret_cast<const float2*>(xrow);
#pragma unroll
    for (int cc = 0; cc < 9; ++cc) {
        const int c = (half ? 9 : 0) + cc;                      // 4-k chunk; 16 holds k = 64, 65 and zeros, 17 zeros
        float2 x = make_float2(0.0f, 0.0f), y = make_float2(0.0f, 0.0f);
        if (2 * c < N_IN / 2) x = src[2 * c];
        if (2 * c + 1 < N_IN / 2) y = src[2 * c + 1];
        float hx, hy, hz, hw, lx, ly, lz, lw;
        tf32_split<NEAREST>(x.x, hx, lx); tf32_split<NEAREST>(x.y, hy, ly);
        tf32_split<NEAREST>(y.x, hz, lz); tf32_split<NEAREST>(y.y, hw, lw);
        tmem_st4(t_hi + 4 * c, hx, hy, hz, hw);
        tmem_st4(t_lo + 4 * c, lx, ly, lz, lw);
    }
}

// The output stage of k_predict and k_predict_mlp, run by their 256 epilogue threads (etid = 0..255: two per env row,
// column halves; TMEM lane quarter = warp % 4) once the tile's 33 output accumulators (fp32, TMEM columns acc..acc+32)
// are complete: tcgen05.ld, then arrive on `bar_free` (the accumulator may be overwritten), add the bias, evaluate the
// slack penalty (fp64, only for rows that leave the limits), stage Vhat in `out` and write the tile with ONE bulk store
// per destination into the dense output and/or the replay ring at (pos + env) mod capacity (a wrapping or unaligned
// segment falls back to a coalesced store loop).  P: a parameter block with the output fields of PredParams.
template <class P>
__device__ __forceinline__ void predict_epilogue(const P& prm, int64_t tile, int rows, uint32_t acc, uint32_t bar_free,
                                                 const float* bias, float* out, double* pen_part, int etid, int warp) {
    const int ehalf = etid >> 7, row = etid & (PRED_M - 1);
    const double neg_vmax = -prm.v_max;
    // TMEM lane = env row; a warp may only touch the lane quarter 32 * (warp % 4): the first four epilogue warps take
    // columns 0..16 of their quarter, the last four columns 17..32
    const int c0 = ehalf ? 17 : 0;
    const uint32_t taddr = acc + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)c0;
    float r0[16], r1 = 0.0f;
    tmem_ld16(taddr, r0);
    if (ehalf == 0) tmem_ld1(taddr + 16, r1);
    tmem_wait_ld();
    tc_fence_before();
    mbar_arrive(bar_free);                       // the accumulator may be overwritten (tile k + 2)
    if (etid == 0) bulk_wait_read();             // the previous tile's bulk stores have read `out`
    group_sync<2, EPI_THREADS>();                // ... and so have its store loops: `out` is free
    double pen = 0.0;
    if (row < rows) {
        float V[17];
        float vmn = INFINITY, vmx = -INFINITY;
#pragma unroll
        for (int i = 0; i < 17; ++i) {
            if (i < 16 || ehalf == 0) {
                V[i] = (i < 16 ? r0[i < 16 ? i : 0] : r1) + bias[c0 + i];
                out[row * N_OUT + c0 + i] = V[i];
                vmn = fminf(vmn, V[i]); vmx = fmaxf(vmx, V[i]);
            }
        }
        // in-limit voltages (the common case) contribute exactly zero, and the fp32 tests are EXACT
        // (lo_f is the smallest float >= v_min, hi_f the largest <= v_max, V is a float): the fp64 terms
        // are only evaluated for a row that leaves the limits, selected per column by the fp32 test
        if (vmn < prm.lo_f || vmx > prm.hi_f) {
#pragma unroll
            for (int i = 0; i < 17; ++i) {
                if (i < 16 || ehalf == 0) {
                    // v_min - V or V - v_max as ONE fused multiply-add with selected operands (the same
                    // single rounding as the subtraction): a third of the fp64 work of computing both
                    const bool un = V[i] < prm.lo_f, ov = V[i] > prm.hi_f;
                    const double sg = un ? -1.0 : (ov ? 1.0 : 0.0);
                    const double cc = un ? prm.v_min : (ov ? neg_vmax : 0.0);
                    pen = pen + fma(sg, (double)V[i], cc);
                }
            }
        }
    }
    pen_part[ehalf * PRED_M + row] = pen;
    fence_proxy_async();                                 // `out` is read by the bulk stores (async proxy)
    group_sync<2, EPI_THREADS>();                        // the tile's Vhat rows and penalty halves are staged
    const int64_t e = tile * PRED_M + row;
    if (ehalf == 0 && row < rows) {
        const double pw = prm.w * (pen_part[row] + pen_part[PRED_M + row]);
        if (prm.penalty != nullptr) prm.penalty[e] = pw;
        if (prm.ring_pen != nullptr) {               // pos < cap and n <= cap: one conditional subtraction wraps
            const int64_t rr = prm.ring_pos + e;
            prm.ring_pen[rr >= prm.ring_cap ? rr - prm.ring_cap : rr] = (float)pw;
        }
    }

    // ---- coalesced row stores: dense output and/or replay ring (wraps at capacity)
    // (the tile's rows are contiguous in the dense output; in the ring they are contiguous up to
    //  one wrap, so element i of the tile lands at i + base, minus the ring size past the end)
    const int64_t e0 = tile * PRED_M;
    const int64_t ring_elems = prm.ring_cap * N_OUT, ring_base = (prm.ring_pos + e0) * N_OUT;
    const int n_el = rows * N_OUT;
    float* dense = prm.vhat != nullptr ? prm.vhat + e0 * N_OUT : nullptr;
    // 16-byte stores where the destination allows it: a full tile is 1056 float4 (e0 * 33 * 4 bytes is
    // a multiple of 16); the ring segment qualifies when it does not wrap and starts 16-byte aligned
    const bool ring_vec = prm.ring_vhat != nullptr && ((ring_base & 3) == 0) && (ring_base + n_el <= ring_elems);
    if ((n_el & 3) == 0 && (dense == nullptr || ((reinterpret_cast<uintptr_t>(dense) & 15) == 0)) &&
        (prm.ring_vhat == nullptr || (ring_vec && ((reinterpret_cast<uintptr_t>(prm.ring_vhat) & 15) == 0)))) {
        // one bulk store (TMA engine) per destination: the staged tile is the contiguous image of its rows
        if (etid == 0) {
            if (dense != nullptr) bulk_s2g(dense, out, (uint32_t)n_el * 4u);
            if (prm.ring_vhat != nullptr) bulk_s2g(prm.ring_vhat + ring_base, out, (uint32_t)n_el * 4u);
            bulk_commit();
        }
    } else {
        for (int i = etid; i < n_el; i += EPI_THREADS) {
            const float v = out[i];
            if (dense != nullptr) dense[i] = v;
            if (prm.ring_vhat != nullptr) {
                int64_t o = ring_base + i;
                o = o >= ring_elems ? o - ring_elems : o;
                prm.ring_vhat[o] = v;
            }
        }
    }
}

__global__ void __launch_bounds__(PRED_THREADS, 1) k_predict(const PredParams prm) {
    extern __shared__ __align__(128) uint8_t smem[];
    float* Bsm = reinterpret_cast<float*>(smem + OFF_BHI);              // hi then lo, contiguous
    float* out = reinterpret_cast<float*>(smem + OFF_OUT);
    float* bias = reinterpret_cast<float*>(smem + OFF_BIAS);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + OFF_TMEM);
    double* pen_part = reinterpret_cast<double*>(smem + OFF_PEN);
    const uint32_t bar_full0 = smem_u32(smem + OFF_BAR), bar_mma0 = bar_full0 + 8 * N_STAGES, bar_free0 = bar_mma0 + 16,
                   bar_w = bar_free0 + 16, bar_a0 = bar_w + 8;
    const int tid = threadIdx.x, warp = __shfl_sync(0xFFFFFFFFu, tid >> 5, 0);   // warp-uniform for the compiler
    const int row = tid & (PRED_M - 1);                                 // env row of the tile (both groups)
    const int64_t n_tiles = (prm.n + PRED_M - 1) / PRED_M;

    auto rows_of = [&](int64_t tl) -> int { const int64_t r = prm.n - tl * PRED_M; return (int)(r < PRED_M ? r : PRED_M); };
    auto tma_ok = [&](int64_t tl) -> bool { return ((rows_of(tl) * N_IN * 4) & 15) == 0; };
    // this CTA's tiles: blockIdx.x + k * gridDim.x, k = 0 .. n_my - 1 (the grid never exceeds the tile count)
    const int n_my = (int)((n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x);
    auto tile_of = [&](int k) -> int64_t { return (int64_t)blockIdx.x + (int64_t)k * gridDim.x; };

    auto issue = [&](int k) {                                           // one thread only (MMA warp)
        const int64_t tl = tile_of(k);
        if (!tma_ok(tl)) return;                                        // odd-sized last tile: plain loads by the producers
        const uint32_t bytes = (uint32_t)(rows_of(tl) * N_IN * 4);
        const int s = k % N_STAGES;
        const uint32_t bar = bar_full0 + 8 * s;
        mbar_expect_tx(bar, bytes);
        tma_load_1d(smem_u32(smem + OFF_STAGE + s * STAGE_BYTES), prm.X + tl * (int64_t)(PRED_M * N_IN), bytes, bar);
    };
    // ---- one-time setup: barriers, TMEM, weights; the first TMA loads are issued before anything else
    if (tid == 0) {
        for (int s = 0; s < N_STAGES; ++s) mbar_init(bar_full0 + 8 * s, 1);
        mbar_init(bar_mma0, 1); mbar_init(bar_mma0 + 8, 1);
        mbar_init(bar_free0, EPI_THREADS); mbar_init(bar_free0 + 8, EPI_THREADS);
        mbar_init(bar_w, 1);
        mbar_init(bar_a0, PROD_THREADS); mbar_init(bar_a0 + 8, PROD_THREADS);
        mbar_init_fence();
        mbar_expect_tx(bar_w, 2 * B_BYTES);                             // weights: one bulk copy, awaited before the first MMA
        tma_load_1d(smem_u32(Bsm), prm.B, 2 * B_BYTES, bar_w);
        for (int k = 0; k < N_STAGES && k < n_my; ++k) issue(k);        // the first X tiles travel during the rest of the setup
    }
    if (warp == 0) {
        tmem_alloc<TMEM_COLS>(smem_u32(tmem_slot));
        tmem_relinquish();
    }
    if (tid < PRED_N) bias[tid] = prm.bias[tid];
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // one tile's MMAs: 9 k-steps x 3 products (hi*hi + lo*hi + hi*lo), A from TMEM buffer `ab`
    auto mma_tile = [&](uint32_t acc, uint32_t ab) {
        const uint32_t b_hi = smem_u32(Bsm), b_lo = b_hi + B_BYTES;
        const uint32_t t_hi = tmem_base + A_COL0 + ab * A_COLS, t_lo = t_hi + PRED_K;
#pragma unroll
        for (int ks = 0; ks < PRED_K / 8; ++ks) {
            const uint32_t bo = ks * 2 * (PRED_N * 16);
            const uint64_t dbh = umma_desc(b_hi + bo, PRED_N * 16, 128), dbl = umma_desc(b_lo + bo, PRED_N * 16, 128);
            umma_tf32_ts(acc, t_hi + 8 * ks, dbh, IDESC, ks > 0 ? 1u : 0u);
            umma_tf32_ts(acc, t_lo + 8 * ks, dbh, IDESC, 1u);
            umma_tf32_ts(acc, t_hi + 8 * ks, dbl, IDESC, 1u);
        }
    };

    if (warp == MMA_WARP) {
        // =============================================================== MMA warp: TMA issue, tcgen05.mma issue
        for (int k = 0; k < n_my; ++k) {
            const int b = k & 1;
            mbar_wait(bar_a0 + 8 * b, (uint32_t)((k >> 1) & 1));        // A buffer b holds tile k; its staging buffer is read
            if (k >= 2) mbar_wait(bar_free0 + 8 * b, (uint32_t)(((k >> 1) - 1) & 1));   // epilogue of tile k - 2 drained the accumulator
            if (k == 0) mbar_wait(bar_w, 0u);                           // the weights have landed
            tc_fence_after();
            __syncwarp();
            if (elect_one()) {
                mma_tile(tmem_base + (uint32_t)b * ACC_COLS, (uint32_t)b);
                umma_commit(bar_mma0 + 8 * b);
                if (k + N_STAGES < n_my) issue(k + N_STAGES);           // refill the staging buffer, N_STAGES tiles ahead -- AFTER the MMAs:
                                                                        // issuing the bulk copy first delays them by its issue latency
                                                                        // (k_policy: 315 -> 266 us from this order alone)
            }
            __syncwarp();
        }
    } else if (warp < PROD_THREADS / 32) {
        // =============================================================== producers: 3xTF32 split -> A operand in TMEM
        // thread = (env row, K half); a warp writes the TMEM lane quarter 32 * (warp % 4) = its rows
        const int half = tid >> 7;
        for (int k = 0; k < n_my; ++k) {
            const int s = k % N_STAGES, b = k & 1;
            const int64_t tile = tile_of(k);
            const int rows = rows_of(tile);
            float* stage = reinterpret_cast<float*>(smem + OFF_STAGE + s * STAGE_BYTES);
            if (tma_ok(tile)) {
                mbar_wait(bar_full0 + 8 * s, (uint32_t)((k / N_STAGES) & 1));
            } else {
                const float* src = prm.X + tile * (int64_t)(PRED_M * N_IN);
                for (int i = tid; i < rows * N_IN; i += PROD_THREADS) stage[i] = src[i];
                group_sync<1, PROD_THREADS>();
            }
            // the MMAs of tile k - 2 have read A buffer b
            if (k >= 2) mbar_wait(bar_mma0 + 8 * b, (uint32_t)(((k >> 1) - 1) & 1));
            tc_fence_after();
            const uint32_t t_hi = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + A_COL0 + (uint32_t)b * A_COLS;
            // rows past the end of a partial tile split whatever the staging buffer holds: never stored
            split_x_to_tmem<false>(stage + row * N_IN, half, t_hi, t_hi + PRED_K);
            tmem_wait_st();
            tc_fence_before();
            mbar_arrive(bar_a0 + 8 * b);
        }
    } else if (warp < (PROD_THREADS + EPI_THREADS) / 32) {
        // =============================================================== epilogue: TMEM -> bias, penalty -> ring
        const int etid = tid - PROD_THREADS;
        for (int k = 0; k < n_my; ++k) {
            const int b = k & 1;
            const int64_t tile = tile_of(k);
            mbar_wait(bar_mma0 + 8 * b, (uint32_t)((k >> 1) & 1));
            tc_fence_after();
            predict_epilogue(prm, tile, rows_of(tile), tmem_base + (uint32_t)b * ACC_COLS, bar_free0 + 8 * b, bias, out, pen_part,
                             etid, warp);
        }
        if (etid == 0) bulk_wait_all();                  // shared memory must outlive the bulk stores
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<TMEM_COLS>(tmem_base);
}

// ---------------------------------------------------------------------------- k_predict_mlp
// scikit-learn MLPRegressor semantics: h_0 = x (66), h_l = act(W_l h_{l-1} + b_l) for the 1..3 hidden layers,
// Vhat = W_L h_{L-1} + b_L (identity output, 33).  The same warp roles, tiles and epilogue as k_predict; every layer
// is a tcgen05.mma (kind::tf32, M = 128, N = the layer's padded width, 3xTF32) with its A operand in TMEM:
//   MMA warp 16   X bulk copies (n_stages >= 2 staging buffers), then per tile one MMA group per layer, each
//                 issued when the producers have written that layer's A operand
//   producers     layer 1: the split of k_predict (split_x_to_tmem); each hidden layer: tcgen05.ld of the hidden
//   (warps 0-7)   accumulator, + bias, activation (fp32, accurate functions), 3xTF32 split, tcgen05.st into the A
//                 region, which the next layer's MMA reads (two threads per row: column halves)
//   epilogue      predict_epilogue on the output accumulator (two of them, so the epilogue of tile k overlaps tile k+1)
// The split weights of every layer stay in shared memory for the CTA's lifetime ([layer][hi | lo][k-chunk][n][4],
// one bulk copy).  TMEM: output accumulators at columns 0 and 64, the hidden accumulator at 128 (h_cols = the widest
// padded hidden layer), the A region after it (hi K | lo K, K = 72 or a padded hidden width).  The host plans both
// (mlp_plan) and accepts a model only if they fit.
constexpr int MLP_MAX_LAYERS = 4, MLP_MAX_WIDTH = 128, MLP_MAX_STAGES = 5;
constexpr uint32_t MLP_OFF_OUT = 0;                                           // [128][33] fp32 Vhat staging
constexpr uint32_t MLP_OFF_PEN = MLP_OFF_OUT + PRED_M * N_OUT * 4;            // [2][128] fp64 penalty partials
constexpr uint32_t MLP_OFF_BAR = MLP_OFF_PEN + 2 * PRED_M * 8;                // full[5], out_done[2], out_free[2], weights, a_ready, hid_done
constexpr uint32_t MLP_OFF_TMEM = MLP_OFF_BAR + 12 * 8;
constexpr uint32_t MLP_OFF_BIAS = MLP_OFF_TMEM + 16;                          // padded biases of every layer
constexpr uint32_t MLP_OFF_W = (MLP_OFF_BIAS + MLP_MAX_LAYERS * MLP_MAX_WIDTH * 4 + 127) & ~127u;
constexpr uint32_t SMEM_LIMIT = 227 * 1024;                                   // dynamic shared memory of one block
constexpr uint32_t MLP_HID_COL0 = 2 * ACC_COLS;

struct MlpParams {
    const float* X; int64_t n;
    const float* W; const float* bias;                       // weight image (shared-memory layout), padded biases
    float* vhat; double* penalty;                            // dense outputs (may be null)
    float* ring_vhat; float* ring_pen; int64_t ring_cap, ring_pos;   // replay sink (may be null)
    double v_min, v_max, w;
    float lo_f, hi_f;                                        // smallest float >= v_min, largest float <= v_max
    int n_layers, act, n_stages, h_cols, n_bias;
    uint32_t w_bytes;
    int k_pad[MLP_MAX_LAYERS], n_pad[MLP_MAX_LAYERS];        // per layer: padded input / output width
    uint32_t w_off[MLP_MAX_LAYERS]; int b_off[MLP_MAX_LAYERS];   // per layer: byte offset of its weights, float offset of its bias
};

__device__ __forceinline__ float activate(float z, int act) {
    switch (act) {
        case FP_ACT_RELU: return z < 0.0f ? 0.0f : z;       // NaN propagates, as np.maximum(z, 0)
        case FP_ACT_TANH: return tanhf(z);
        case FP_ACT_LOGISTIC: return 1.0f / (1.0f + expf(-z));
        default: return z;
    }
}

__global__ void __launch_bounds__(PRED_THREADS, 1) k_predict_mlp(const MlpParams prm) {
    extern __shared__ __align__(128) uint8_t smem[];
    float* out = reinterpret_cast<float*>(smem + MLP_OFF_OUT);
    double* pen_part = reinterpret_cast<double*>(smem + MLP_OFF_PEN);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + MLP_OFF_TMEM);
    float* bias = reinterpret_cast<float*>(smem + MLP_OFF_BIAS);
    const uint32_t w_sm = smem_u32(smem + MLP_OFF_W), off_stage = MLP_OFF_W + prm.w_bytes;
    const uint32_t bar_full0 = smem_u32(smem + MLP_OFF_BAR), bar_out0 = bar_full0 + 8 * MLP_MAX_STAGES, bar_free0 = bar_out0 + 16,
                   bar_w = bar_free0 + 16, bar_a = bar_w + 8, bar_hid = bar_a + 8;
    const int n_stages = prm.n_stages, L = prm.n_layers;
    const int tid = threadIdx.x, warp = __shfl_sync(0xFFFFFFFFu, tid >> 5, 0);
    const int row = tid & (PRED_M - 1);
    const int64_t n_tiles = (prm.n + PRED_M - 1) / PRED_M;

    auto rows_of = [&](int64_t tl) -> int { const int64_t r = prm.n - tl * PRED_M; return (int)(r < PRED_M ? r : PRED_M); };
    auto tma_ok = [&](int64_t tl) -> bool { return ((rows_of(tl) * N_IN * 4) & 15) == 0; };
    const int n_my = (int)((n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x);
    auto tile_of = [&](int k) -> int64_t { return (int64_t)blockIdx.x + (int64_t)k * gridDim.x; };
    auto issue = [&](int k) {                                           // one thread only (MMA warp)
        const int64_t tl = tile_of(k);
        if (!tma_ok(tl)) return;                                        // odd-sized last tile: plain loads by the producers
        const uint32_t bytes = (uint32_t)(rows_of(tl) * N_IN * 4);
        const int s = k % n_stages;
        mbar_expect_tx(bar_full0 + 8 * s, bytes);
        tma_load_1d(smem_u32(smem + off_stage + s * STAGE_BYTES), prm.X + tl * (int64_t)(PRED_M * N_IN), bytes, bar_full0 + 8 * s);
    };
    if (tid == 0) {
        for (int s = 0; s < n_stages; ++s) mbar_init(bar_full0 + 8 * s, 1);
        mbar_init(bar_out0, 1); mbar_init(bar_out0 + 8, 1);
        mbar_init(bar_free0, EPI_THREADS); mbar_init(bar_free0 + 8, EPI_THREADS);
        mbar_init(bar_w, 1);
        mbar_init(bar_a, PROD_THREADS);
        mbar_init(bar_hid, 1);
        mbar_init_fence();
        mbar_expect_tx(bar_w, prm.w_bytes);                             // weights: one bulk copy, awaited before the first MMA
        tma_load_1d(w_sm, prm.W, prm.w_bytes, bar_w);
        for (int k = 0; k < n_stages && k < n_my; ++k) issue(k);
    }
    if (warp == 0) {
        tmem_alloc<TMEM_COLS>(smem_u32(tmem_slot));
        tmem_relinquish();
    }
    for (int i = tid; i < prm.n_bias; i += PRED_THREADS) bias[i] = prm.bias[i];
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t t_hid = tmem_base + MLP_HID_COL0, t_a = t_hid + (uint32_t)prm.h_cols;

    if (warp == MMA_WARP) {
        // =============================================================== MMA warp: TMA issue, one MMA group per layer
        uint32_t ph_a = 0;
        for (int k = 0; k < n_my; ++k) {
            const int b = k & 1;
            for (int l = 0; l < L; ++l) {
                const bool last = l == L - 1;
                mbar_wait(bar_a, ph_a); ph_a ^= 1u;                     // layer l's A operand is in TMEM
                if (last && k >= 2) mbar_wait(bar_free0 + 8 * b, (uint32_t)(((k >> 1) - 1) & 1));   // tile k - 2 drained acc b
                if (k == 0 && l == 0) mbar_wait(bar_w, 0u);
                tc_fence_after();
                __syncwarp();
                if (elect_one()) {
                    const int K = prm.k_pad[l], N = prm.n_pad[l];
                    const uint32_t acc = last ? tmem_base + (uint32_t)b * ACC_COLS : t_hid;
                    const uint32_t b_hi = w_sm + prm.w_off[l], b_lo = b_hi + (uint32_t)(K * N * 4);
                    const uint32_t idesc = umma_idesc_tf32(PRED_M, (uint32_t)N);
                    for (int ks = 0; ks < K / 8; ++ks) {               // 3xTF32: hi*hi + lo*hi + hi*lo
                        const uint32_t bo = (uint32_t)(ks * 2 * N * 16);
                        const uint64_t dbh = umma_desc(b_hi + bo, N * 16, 128), dbl = umma_desc(b_lo + bo, N * 16, 128);
                        umma_tf32_ts(acc, t_a + 8 * ks, dbh, idesc, ks > 0 ? 1u : 0u);
                        umma_tf32_ts(acc, t_a + K + 8 * ks, dbh, idesc, 1u);
                        umma_tf32_ts(acc, t_a + 8 * ks, dbl, idesc, 1u);
                    }
                    umma_commit(last ? bar_out0 + 8 * b : bar_hid);
                    if (l == 0 && k + n_stages < n_my) issue(k + n_stages);   // the producers have read tile k's staging buffer
                }
                __syncwarp();
            }
        }
    } else if (warp < PROD_THREADS / 32) {
        // =============================================================== producers: A operand of every layer in TMEM
        const int half = tid >> 7;
        const uint32_t lane = (uint32_t)((warp & 3) * 32) << 16;
        uint32_t ph_hid = 0;
        for (int k = 0; k < n_my; ++k) {
            const int s = k % n_stages;
            const int64_t tile = tile_of(k);
            const int rows = rows_of(tile);
            float* stage = reinterpret_cast<float*>(smem + off_stage + s * STAGE_BYTES);
            if (tma_ok(tile)) {
                mbar_wait(bar_full0 + 8 * s, (uint32_t)((k / n_stages) & 1));
            } else {
                const float* src = prm.X + tile * (int64_t)(PRED_M * N_IN);
                for (int i = tid; i < rows * N_IN; i += PROD_THREADS) stage[i] = src[i];
                group_sync<1, PROD_THREADS>();
            }
            // the output-layer MMAs of tile k - 1 have read the A region
            if (k >= 1) mbar_wait(bar_out0 + 8 * ((k - 1) & 1), (uint32_t)(((k - 1) >> 1) & 1));
            tc_fence_after();
            // rows past the end of a partial tile compute on whatever the staging buffer holds: never stored
            split_x_to_tmem<true>(stage + row * N_IN, half, t_a + lane, t_a + lane + PRED_K);
            tmem_wait_st();
            tc_fence_before();
            mbar_arrive(bar_a);
            for (int l = 0; l < L - 1; ++l) {
                mbar_wait(bar_hid, ph_hid); ph_hid ^= 1u;               // hidden layer l's accumulator is complete
                tc_fence_after();
                const int N = prm.n_pad[l], hc = N / 2, cb = half * hc; // this thread: columns cb .. cb + hc - 1
                const float* bl = bias + prm.b_off[l];
                for (int c0 = 0; c0 < hc; c0 += 32) {
                    float r[4][8];
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (c0 + 8 * j < hc) tmem_ld8(t_hid + lane + (uint32_t)(cb + c0 + 8 * j), r[j]);
                    tmem_wait_ld();
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        if (c0 + 8 * j < hc) {
                            const int c = cb + c0 + 8 * j;
                            float hi[8], lo[8];
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                tf32_split<true>(activate(r[j][i] + bl[c + i], prm.act), hi[i], lo[i]);
                            }
                            // next layer's A: K = N columns, hi at t_a + c, lo at t_a + N + c
                            tmem_st4(t_a + lane + (uint32_t)c, hi[0], hi[1], hi[2], hi[3]);
                            tmem_st4(t_a + lane + (uint32_t)(c + 4), hi[4], hi[5], hi[6], hi[7]);
                            tmem_st4(t_a + lane + (uint32_t)(N + c), lo[0], lo[1], lo[2], lo[3]);
                            tmem_st4(t_a + lane + (uint32_t)(N + c + 4), lo[4], lo[5], lo[6], lo[7]);
                        }
                    }
                }
                tmem_wait_st();
                tc_fence_before();
                mbar_arrive(bar_a);                                     // the accumulator is read, the next A is written
            }
        }
    } else if (warp < (PROD_THREADS + EPI_THREADS) / 32) {
        // =============================================================== epilogue: the output layer, as k_predict
        const int etid = tid - PROD_THREADS;
        const float* b_out = bias + prm.b_off[L - 1];
        for (int k = 0; k < n_my; ++k) {
            const int b = k & 1;
            const int64_t tile = tile_of(k);
            mbar_wait(bar_out0 + 8 * b, (uint32_t)((k >> 1) & 1));
            tc_fence_after();
            predict_epilogue(prm, tile, rows_of(tile), tmem_base + (uint32_t)b * ACC_COLS, bar_free0 + 8 * b, b_out, out, pen_part,
                             etid, warp);
        }
        if (etid == 0) bulk_wait_all();                  // shared memory must outlive the bulk stores
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<TMEM_COLS>(tmem_base);
}

// ---------------------------------------------------------------------------- replay ring
// n consecutive ring rows starting at `pos` are contiguous in memory up to one wrap, so both
// copies are flat, fully coalesced and free of integer division: element i <-> ring element
// pos * width + i, minus the ring size past the end.
__global__ void k_replay_write(float* __restrict__ dst, int64_t cap, int width, int64_t pos, int64_t n,
                               const float* __restrict__ src) {
    const int64_t total = n * width, ring = cap * width, base = pos * width;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t o = base + i;
        o = o >= ring ? o - ring : o;
        dst[o] = src[i];
    }
}

__global__ void k_replay_gather(const float* __restrict__ field, int64_t cap, int width, int64_t first, int64_t batch,
                                float* __restrict__ out) {
    const int64_t total = batch * width, ring = cap * width, base = first * width;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t o = base + i;
        o = o >= ring ? o - ring : o;
        out[i] = field[o];
    }
}

// Input, outputs and replay sink of fp_predict / fp_predict_mlp into the kernel's parameter block P (PredParams or
// MlpParams): the checks and messages of both entry points.
template <class P>
int bind_outputs(FpHandle* h, const char* what, P& prm, int64_t n, const float* d_X, float* d_vhat, double* d_penalty,
                 FpReplay* sink, int32_t f_vhat, int32_t f_penalty, int64_t pos, double v_min, double v_max, double w) {
    const std::string fn(what);
    if (n < 1 || !d_X) return fail(h, FP_EINVAL, fn + ": bad arguments");
    if (((uintptr_t)d_X & 15) != 0) return fail(h, FP_EINVAL, fn + ": X must be 16-byte aligned (TMA)");
    prm.X = d_X; prm.n = n; prm.vhat = d_vhat; prm.penalty = d_penalty;
    prm.v_min = v_min; prm.v_max = v_max; prm.w = w;
    prm.lo_f = (float)v_min; if ((double)prm.lo_f < v_min) prm.lo_f = std::nextafterf(prm.lo_f, INFINITY);
    prm.hi_f = (float)v_max; if ((double)prm.hi_f > v_max) prm.hi_f = std::nextafterf(prm.hi_f, -INFINITY);
    prm.ring_cap = 1; prm.ring_pos = 0;
    if (sink) {
        const int nf = (int)sink->widths.size();
        if (n > sink->capacity || pos < 0 || pos >= sink->capacity)
            return fail(h, FP_EINVAL, fn + ": rows do not fit the replay ring");
        if (f_vhat >= 0) {
            if (f_vhat >= nf || sink->widths[f_vhat] != N_OUT) return fail(h, FP_EINVAL, fn + ": Vhat field must have width 33");
            prm.ring_vhat = sink->d_fields[f_vhat];
        }
        if (f_penalty >= 0) {
            if (f_penalty >= nf || sink->widths[f_penalty] != 1) return fail(h, FP_EINVAL, fn + ": penalty field must have width 1");
            prm.ring_pen = sink->d_fields[f_penalty];
        }
        prm.ring_cap = sink->capacity; prm.ring_pos = pos;
    }
    return FP_OK;
}

// x rounded to the nearest TF32 value, ties away from zero (cvt.rna.tf32.f32 of the kernel's split); x finite
float tf32_nearest(float x) {
    uint32_t u; std::memcpy(&u, &x, 4);
    u = (u + 0x1000u) & 0xFFFFE000u;
    std::memcpy(&x, &u, 4);
    return x;
}

// Persistent grid: one CTA per SM at most, never more CTAs than 128-env tiles.
cudaError_t grid_of(const FpHandle* h, int64_t n, int* grid) {
    int sms = 0;
    const cudaError_t e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
    const int64_t tiles = (n + PRED_M - 1) / PRED_M;
    *grid = (int)(tiles < sms ? tiles : sms);
    return e;
}

}  // namespace

void predictor_free(PredictorState* p) {
    if (!p) return;
    cudaFree(p->d_B); cudaFree(p->d_bias);
    p->d_B = nullptr; p->d_bias = nullptr; p->loaded = 0;
}

void mlp_free(MlpState* m) {
    if (!m) return;
    cudaFree(m->d_W); cudaFree(m->d_bias);
    m->d_W = nullptr; m->d_bias = nullptr; m->loaded = 0;
}

extern "C" {

int fp_predictor_load(FpHandle* h, int32_t n_in, int32_t n_out, const double* h_A, const double* h_c, double v_min,
                      double v_max, double slack_weight) {
    if (!h) return FP_EINVAL;
    if (n_in != N_IN || n_out != N_OUT || !h_A || !h_c)
        return fail(h, FP_EINVAL, "fp_predictor_load: expects a 66 -> 33 affine model (2*n_bus inputs, n_bus outputs)");
    PredictorState* p = &h->pred;
    USE_DEVICE(h);
    predictor_free(p);                             // clears p->loaded: set again only after the last step below
    // weights: fp64 -> (hi, lo) TF32-representable pair, UMMA K-major layout [part][k-chunk][n][4], zero padded
    std::vector<float> B(2 * PRED_KC * PRED_N * 4, 0.0f), bias(PRED_N, 0.0f);
    for (int n = 0; n < N_OUT; ++n) {
        for (int k = 0; k < N_IN; ++k) {
            const double a = h_A[(size_t)n * N_IN + k];
            float hi = (float)a;
            uint32_t u; std::memcpy(&u, &hi, 4); u &= 0xFFFFE000u; std::memcpy(&hi, &u, 4);
            const float lo = (float)(a - (double)hi);
            const size_t off = ((size_t)(k >> 2) * PRED_N + n) * 4 + (k & 3);
            B[off] = hi; B[(size_t)PRED_KC * PRED_N * 4 + off] = lo;
        }
        bias[n] = (float)h_c[n];
    }
    CUDA_TRY(h, alloc_group({{&p->d_B, B.size() * 4}, {&p->d_bias, bias.size() * 4}}));
    CUDA_TRY(h, cudaMemcpy(p->d_B, B.data(), B.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(p->d_bias, bias.data(), bias.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaFuncSetAttribute(k_predict, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
    p->n_in = n_in; p->n_out = n_out; p->v_min = v_min; p->v_max = v_max; p->slack_weight = slack_weight;
    p->loaded = 1;
    return FP_OK;
}

int fp_predict(FpHandle* h, int64_t n, const float* d_X, float* d_vhat, double* d_penalty, FpReplay* sink,
               int32_t f_vhat, int32_t f_penalty, int64_t pos, void* stream) {
    if (!h) return FP_EINVAL;
    const PredictorState* p = &h->pred;
    if (!p->loaded) return fail(h, FP_ESTATE, "fp_predict: call fp_predictor_load first");
    PredParams prm;
    std::memset(&prm, 0, sizeof(prm));
    prm.B = p->d_B; prm.bias = p->d_bias;
    if (const int rc = bind_outputs(h, "fp_predict", prm, n, d_X, d_vhat, d_penalty, sink, f_vhat, f_penalty, pos, p->v_min,
                                    p->v_max, p->slack_weight))
        return rc;
    USE_DEVICE(h);
    int grid = 0;
    CUDA_TRY(h, grid_of(h, n, &grid));
    k_predict<<<grid, PRED_THREADS, SMEM_BYTES, (cudaStream_t)stream>>>(prm);
    return launched(h, "k_predict");
}

int fp_predictor_load_mlp(FpHandle* h, int32_t n_layers, const int32_t* h_widths, const double* h_W, const double* h_b,
                          int32_t activation, double v_min, double v_max, double slack_weight) {
    if (!h) return FP_EINVAL;
    if (n_layers < 2 || n_layers > MLP_MAX_LAYERS || !h_widths || !h_W || !h_b)
        return fail(h, FP_EINVAL, "fp_predictor_load_mlp: expects 1 to 3 hidden layers (n_layers 2..4) and non-null widths, weights, biases");
    if (h_widths[0] != N_IN || h_widths[n_layers] != N_OUT)
        return fail(h, FP_EINVAL, "fp_predictor_load_mlp: input width must be 66 (2*n_bus) and output width 33 (n_bus)");
    for (int l = 1; l < n_layers; ++l)
        if (h_widths[l] < 1 || h_widths[l] > MLP_MAX_WIDTH)
            return fail(h, FP_EINVAL, "fp_predictor_load_mlp: hidden widths must be 1..128");
    if (activation < FP_ACT_IDENTITY || activation > FP_ACT_LOGISTIC)
        return fail(h, FP_EINVAL, "fp_predictor_load_mlp: unknown activation (FP_ACT_IDENTITY, _RELU, _TANH, _LOGISTIC)");
    if (!(v_min < v_max) || !(slack_weight > 0.0))
        return fail(h, FP_EINVAL, "fp_predictor_load_mlp: v_min < v_max and slack_weight > 0 required");
    // plan: layer l is [n_pad][k_pad] (N padded to 16 for UMMA, K to 8; a hidden layer's K is the padded width of
    // the layer before, whose padding units are act(0) times zero weights)
    MlpState m;
    m.n_layers = n_layers; m.act = activation;
    size_t n_w = 0, n_b = 0;
    for (int l = 0; l < n_layers; ++l) {
        m.k_pad[l] = l == 0 ? PRED_K : m.n_pad[l - 1];
        m.n_pad[l] = (h_widths[l + 1] + 15) / 16 * 16;
        m.w_off[l] = m.w_bytes;
        m.b_off[l] = m.n_bias;
        m.w_bytes += (uint32_t)(2 * m.k_pad[l] * m.n_pad[l] * 4);
        m.n_bias += m.n_pad[l];
        if (l < n_layers - 1) m.h_cols = std::max(m.h_cols, m.n_pad[l]);
        n_w += (size_t)h_widths[l + 1] * h_widths[l];
        n_b += (size_t)h_widths[l + 1];
    }
    for (size_t i = 0; i < n_w; ++i)
        if (!std::isfinite(h_W[i])) return fail(h, FP_EINVAL, "fp_predictor_load_mlp: non-finite weight");
    for (size_t i = 0; i < n_b; ++i)
        if (!std::isfinite(h_b[i])) return fail(h, FP_EINVAL, "fp_predictor_load_mlp: non-finite bias");
    const uint32_t fixed = MLP_OFF_W + m.w_bytes;
    m.n_stages = fixed >= SMEM_LIMIT ? 0 : std::min<int>(MLP_MAX_STAGES, (int)((SMEM_LIMIT - fixed) / STAGE_BYTES));
    if (m.n_stages < 2)
        return fail(h, FP_EINVAL, "fp_predictor_load_mlp: the model needs " + std::to_string(m.w_bytes) +
                                      " bytes of split-TF32 weights; with the output staging, the barriers and two 33 KB X "
                                      "staging buffers that is " + std::to_string(fixed + 2 * STAGE_BYTES) +
                                      " bytes, over the 227 KB (" + std::to_string(SMEM_LIMIT) + " bytes) shared-memory limit of one block");
    m.smem_bytes = fixed + (uint32_t)m.n_stages * STAGE_BYTES;
    const int tmem_cols = (int)MLP_HID_COL0 + m.h_cols + 2 * std::max(PRED_K, m.h_cols);
    if (tmem_cols > (int)TMEM_COLS)
        return fail(h, FP_EINVAL, "fp_predictor_load_mlp: the TMEM plan needs " + std::to_string(tmem_cols) + " of 512 columns");
    // weights: fp64 -> (hi, lo) TF32 values rounded to nearest, per layer, UMMA K-major layout [part][k-chunk][n][4], zero padded
    std::vector<float> W(m.w_bytes / 4, 0.0f), bias(m.n_bias, 0.0f);
    const double* wl = h_W;
    const double* bl = h_b;
    for (int l = 0; l < n_layers; ++l) {
        const int n_in = h_widths[l], n_out = h_widths[l + 1], N = m.n_pad[l];
        float* hi_part = W.data() + m.w_off[l] / 4;
        float* lo_part = hi_part + (size_t)m.k_pad[l] * N;
        for (int n = 0; n < n_out; ++n) {
            for (int k = 0; k < n_in; ++k) {
                const double a = wl[(size_t)n * n_in + k];
                const float hi = tf32_nearest((float)a);
                const size_t off = ((size_t)(k >> 2) * N + n) * 4 + (k & 3);
                hi_part[off] = hi; lo_part[off] = tf32_nearest((float)(a - (double)hi));
            }
            bias[m.b_off[l] + n] = (float)bl[n];
        }
        wl += (size_t)n_out * n_in;
        bl += n_out;
    }
    MlpState* dst = &h->mlp;
    USE_DEVICE(h);
    mlp_free(dst);                                 // clears dst->loaded: set again only after the last step below
    CUDA_TRY(h, alloc_group({{&m.d_W, W.size() * 4}, {&m.d_bias, bias.size() * 4}}));
    dst->d_W = m.d_W; dst->d_bias = m.d_bias;       // owned by the slot from here on (freed by mlp_free / fp_destroy)
    CUDA_TRY(h, cudaMemcpy(m.d_W, W.data(), W.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(m.d_bias, bias.data(), bias.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaFuncSetAttribute(k_predict_mlp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_LIMIT));
    m.v_min = v_min; m.v_max = v_max; m.slack_weight = slack_weight;
    m.loaded = 1;
    *dst = m;
    return FP_OK;
}

int fp_predict_mlp(FpHandle* h, int64_t n, const float* d_X, float* d_vhat, double* d_penalty, FpReplay* sink,
                   int32_t f_vhat, int32_t f_penalty, int64_t pos, void* stream) {
    if (!h) return FP_EINVAL;
    const MlpState* m = &h->mlp;
    if (!m->loaded) return fail(h, FP_ESTATE, "fp_predict_mlp: call fp_predictor_load_mlp first");
    MlpParams prm;
    std::memset(&prm, 0, sizeof(prm));
    prm.W = m->d_W; prm.bias = m->d_bias;
    prm.n_layers = m->n_layers; prm.act = m->act; prm.n_stages = m->n_stages; prm.h_cols = m->h_cols; prm.n_bias = m->n_bias;
    prm.w_bytes = m->w_bytes;
    for (int l = 0; l < MLP_MAX_LAYERS; ++l) {
        prm.k_pad[l] = m->k_pad[l]; prm.n_pad[l] = m->n_pad[l]; prm.w_off[l] = m->w_off[l]; prm.b_off[l] = m->b_off[l];
    }
    if (const int rc = bind_outputs(h, "fp_predict_mlp", prm, n, d_X, d_vhat, d_penalty, sink, f_vhat, f_penalty, pos, m->v_min,
                                    m->v_max, m->slack_weight))
        return rc;
    USE_DEVICE(h);
    int grid = 0;
    CUDA_TRY(h, grid_of(h, n, &grid));
    k_predict_mlp<<<grid, PRED_THREADS, m->smem_bytes, (cudaStream_t)stream>>>(prm);
    return launched(h, "k_predict_mlp");
}

// ------------------------------------------------------------------ replay ring (TransReplayBuffer)
int fp_replay_create(int64_t capacity, int32_t n_fields, const int32_t* widths, int device, FpReplay** out) {
    if (!out || capacity < 1 || n_fields < 1 || n_fields > 64 || !widths) return fail<FpReplay>(nullptr, FP_EINVAL, "fp_replay_create: bad arguments");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return fail<FpReplay>(nullptr, FP_ECUDA, "fp_replay_create: no CUDA device (there is no CPU fallback)");
    if (device < 0 || device >= ndev) return fail<FpReplay>(nullptr, FP_EINVAL, "fp_replay_create: bad device index");
    for (int f = 0; f < n_fields; ++f)
        if (widths[f] < 1) return fail<FpReplay>(nullptr, FP_EINVAL, "fp_replay_create: field width must be >= 1");
    FpReplay* r = new FpReplay();
    r->capacity = capacity; r->device = device;
    const DeviceGuard on_device(device);
    cudaError_t e = on_device.error();
    for (int f = 0; f < n_fields && e == cudaSuccess; ++f) {
        float* p = nullptr;
        if ((e = cudaMalloc(&p, (size_t)capacity * widths[f] * 4)) != cudaSuccess) break;
        r->widths.push_back(widths[f]); r->d_fields.push_back(p);
        e = cudaMemset(p, 0, (size_t)capacity * widths[f] * 4);
    }
    if (e != cudaSuccess) {
        fp_replay_destroy(r);
        return fail<FpReplay>(nullptr, e == cudaErrorMemoryAllocation ? FP_ENOMEM : FP_ECUDA, std::string("fp_replay_create: ") + cudaGetErrorString(e));
    }
    *out = r;
    return FP_OK;
}

int fp_replay_destroy(FpReplay* r) {
    if (!r) return FP_OK;
    const DeviceGuard on_device(r->device);       // best effort: the ring is freed whatever happens
    for (float* p : r->d_fields) cudaFree(p);
    delete r;
    return FP_OK;
}

const char* fp_replay_last_error(const FpReplay* r) { return r ? r->err.c_str() : create_error<FpReplay>().c_str(); }
int64_t fp_replay_len(const FpReplay* r) { return r ? r->len : 0; }
int64_t fp_replay_capacity(const FpReplay* r) { return r ? r->capacity : 0; }
int fp_replay_clear(FpReplay* r) { if (!r) return FP_EINVAL; r->head = 0; r->len = 0; return FP_OK; }     // :29-30

// add_experience (:23-27) for n rows at once: the oldest rows are overwritten when the ring is full
int fp_replay_reserve(FpReplay* r, int64_t n, int64_t* pos) {
    if (!r || !pos) return FP_EINVAL;
    if (n < 1 || n > r->capacity) return fail(r, FP_EINVAL, "fp_replay_reserve: 1 <= n <= capacity required");
    *pos = r->head;
    r->head = (r->head + n) % r->capacity;
    r->len = (r->len + n < r->capacity) ? r->len + n : r->capacity;
    return FP_OK;
}

int fp_replay_write(FpReplay* r, int32_t field, int64_t pos, int64_t n, const float* d_src, void* stream) {
    if (!r) return FP_EINVAL;
    if (field < 0 || field >= (int)r->widths.size() || !d_src || n < 1 || n > r->capacity || pos < 0 || pos >= r->capacity)
        return fail(r, FP_EINVAL, "fp_replay_write: bad arguments");
    USE_DEVICE(r);
    const int w = r->widths[field];
    k_replay_write<<<grid_for(n * w), 256, 0, (cudaStream_t)stream>>>(r->d_fields[field], r->capacity, w, pos, n, d_src);
    CUDA_TRY(r, cudaGetLastError());
    return FP_OK;
}

// get_batch (:14-21): `batch` consecutive rows from logical index `start` (0 = oldest)
int fp_replay_sample(FpReplay* r, int64_t start, int64_t batch, float* const* d_out, void* stream) {
    if (!r || !d_out) return FP_EINVAL;
    if (batch < 1 || start < 0 || start + batch > r->len) return fail(r, FP_EINVAL, "fp_replay_sample: window outside the stored rows");
    USE_DEVICE(r);
    const int64_t first = ((r->head - r->len + start) % r->capacity + r->capacity) % r->capacity;
    for (size_t f = 0; f < r->widths.size(); ++f) {
        if (!d_out[f]) continue;
        const int w = r->widths[f];
        k_replay_gather<<<grid_for(batch * w), 256, 0, (cudaStream_t)stream>>>(r->d_fields[f], r->capacity, w, first, batch, d_out[f]);
    }
    CUDA_TRY(r, cudaGetLastError());
    return FP_OK;
}

int fp_replay_field_ptr(FpReplay* r, int32_t field, float** d_ptr) {
    if (!r || !d_ptr || field < 0 || field >= (int)r->widths.size()) return FP_EINVAL;
    *d_ptr = r->d_fields[field];
    return FP_OK;
}

}  // extern "C"
