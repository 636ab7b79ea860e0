// policy.cu -- the acting policy of the rollout loop on tcgen05 tensor cores (SURVEY 8f rank 1).
//
//   fp_policy_load / fp_policy_act   replace, for N envs x NA agents (1 .. 5) at once, what train_process does per step
//       (madrl/models/model.py:215-216): prep_obs -> Model.policy (model.py:102-140: agent-id one-hot appended,
//       shared parameters) -> RNNAgent.forward (madrl/agents/rnn_agent.py:24-32: fc1 -> LayerNorm -> ReLU ->
//       GRUCell -> fc2) -> select_action (utils/util.py:50-64, continuous / action_enforcebound: x = mean + std eps,
//       action = tanh(x), log_prob = Normal(mean, std).log_prob(x) - log(1 - action^2 + 1e-6); status 'test':
//       action = tanh(mean)).
//
// Input is the env-minor observation ring the step kernel pushes into (fp_step_ring: ring[24][NA][6][n_pad] fp32):
// a tile is (one agent, 128 consecutive envs), and its 144 x 128 input block -- row k = (ring slot, feature),
// 128 contiguous envs -- arrives with coalesced 16-byte LDGSTS copies; nothing is re-materialised.  The rotation of
// the ring (the newest slot moves every step) is absorbed by the WEIGHTS: fc1 is linear in the observation, so the
// loader prepares the 24 column rotations of W1 once and the kernel stages the one that matches the step's slot.
// The one-hot agent id only selects a column of W1: it is folded into a per-agent bias.
//
// Kernel k_policy: one persistent CTA per SM, 16 worker warps (FOUR threads per (env, agent) row: column quarters) + one
// MMA warp; the matrices (135 KB as TF32, UMMA K-major layout) stay in shared memory for the lifetime of the CTA.
// Per tile, two GEMM phases on tcgen05.mma kind::tf32, M = 128, A OPERAND IN TMEM (a thread owns a row and a TMEM
// lane is a row, so tcgen05.st.32x32b writes the operand without touching shared memory), fp32 accumulators in TMEM:
//     P0  workers: 2xTF32 split of the observation block (x = hi + lo, hi TF32-exact)          -> TMEM cols [0, 288)
//     M1  fc1:  acc1[128][64]  = (Xhi + Xlo) W1^T                  36 MMAs, K = 144                  cols [288, 352)
//     E1  workers: + bias(agent), LayerNorm (four-thread reduction), ReLU, split -> A2; h_in split -> A3  [0, 256)
//     M2  GRU:  rz[128][128] = A2 Wih_rz^T + A3 Whh_rz^T;  gi_n = A2 Wih_n^T;  gh_n = A3 Whh_n^T  128 MMAs  [256, 512)
//         issued in two column halves with a commit each (gate rows permuted by the loader): E2 starts on half 0
//     E2  workers: r, z = sigmoid, n = tanh(gi_n + r gh_n), h' = (1 - z) n + z h -> global; fc2 (64 -> 4: 256 FMAs per
//         row, on the CUDA cores in fp32 with the unrounded weights -- cheaper than a third tensor-core round trip),
//         four-thread reduction, + bias, tanh-Normal sampling (Philox4x32-10 + Box-Muller, or caller-supplied eps)
// The workers' phases and the MMA phases of one tile are serial (one tile fills the 512 TMEM columns: the split
// doubles every A operand); the next tile's observation block travels (LDGSTS) underneath.
// Precision: activations keep fp32 accuracy through the two-term split (hi + lo, both products accumulated in fp32);
// the fc1 / GRU MATRICES are held as TF32 (round-to-nearest, 10-bit mantissa): against torch fp32 with the same
// rounded matrices the means agree to ~1e-6, with arbitrary fp32 weights to ~3e-4 (tests/test_gpu_policy.py states both).
#include <cuda.h>

#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "api_handle.cuh"
#include "flex_common.cuh"
#include "sm100_ptx.cuh"

namespace {

constexpr int POL_M = 128;                 // rows per tile = envs of one agent
constexpr int POL_OBS = 144, POL_HID = 64, POL_ACT = 4, POL_H = 24, POL_F = 6;
// Agents per env: NA = 1 .. 5, a template parameter of every kernel below, dispatched once on the handle's count (the
// five-agent instantiations compile to the code of the single-count kernels they replace).  Shared memory, TMEM and the
// small-array offsets stay sized for five agents: for NA < 5 they are upper bounds.
constexpr int POL_NA_MAX = 5;
constexpr int TPR = 4;                     // worker threads per row (column quarters)
constexpr int N_WORKERS = TPR * POL_M;     // 512
constexpr int N_WRITERS = 96;               // k_policy: three warps that copy the tile's observation block into the Transition's `state` rows
                                            // (640 threads = five allocation groups of four warps: 96 registers per thread stay available)
constexpr int CRIT_THREADS = N_WORKERS + 32 + 96;   // k_critic: the last three warps idle (640-thread CTAs measured 3 % faster than 544)
constexpr int POL_THREADS = N_WORKERS + 32 + N_WRITERS;
constexpr int CPT = POL_HID / TPR;         // hidden columns per thread: 16
constexpr int KPT = POL_OBS / TPR;         // observation inputs per thread: 36
constexpr uint32_t W1_BYTES = POL_OBS * POL_HID * 4;                       // 36 864: [36 kc][64 n][4]
constexpr uint32_t WG_RZ_BYTES = POL_HID * 128 * 4, WG_N_BYTES = POL_HID * 64 * 4;   // [16 kc][N][4]
constexpr uint32_t WG_BYTES = 2 * WG_RZ_BYTES + 2 * WG_N_BYTES;            // 98 304: rz_ih, rz_hh, n_ih, n_hh
// small arrays (floats): b1a[5][64], ln_g[64], ln_b[64], b_rz[128] (-(b_ih + b_hh) log2 e), b_in[64], b_hn[64] (x 2 log2 e), W2[64][4] (fp32, unit-major), b2[4] (+12 pad)
constexpr int V_B1A = 0, V_LNG = 320, V_LNB = 384, V_BRZ = 448, V_BIN = 576, V_BHN = 640, V_W2 = 704, V_B2 = 960, V_FLOATS = 992;
constexpr uint32_t OFF_W1 = 0, OFF_WG = OFF_W1 + W1_BYTES, OFF_VEC = OFF_WG + WG_BYTES;
constexpr uint32_t OFF_STAGE = OFF_VEC + V_FLOATS * 4;                     // [144][128] fp32 = 73 728
constexpr uint32_t OFF_LN = OFF_STAGE + POL_OBS * POL_M * 4;               // [TPR][128 rows] float2 (quarter mean, sum of squared deviations)
constexpr uint32_t OFF_FC = OFF_LN + TPR * POL_M * 8;                      // [TPR][128 rows] float4: fc2 partial sums
constexpr uint32_t OFF_BAR = OFF_FC + TPR * POL_M * 16;                    // a_ready, mma_done, weights, x_full
constexpr uint32_t OFF_TMEM = OFF_BAR + 56;                                // (+ mma_done of the two column halves of the GRU GEMMs, stage_copied)
constexpr uint32_t OFF_Z = (OFF_TMEM + 16 + 15) / 16 * 16;                                // [128 rows] float4: the row's four normals, drawn ahead
constexpr uint32_t POL_SMEM = OFF_Z + POL_M * 16;
static_assert(POL_SMEM <= 227 * 1024, "policy kernel exceeds the shared memory of one SM");
static_assert(OFF_STAGE % 128 == 0 && OFF_WG % 128 == 0 && OFF_VEC % 16 == 0 && (V_FLOATS * 4) % 16 == 0, "operand alignment");
// TMEM columns (512 = the whole TMEM: one CTA per SM)
constexpr uint32_t C_XHI = 0, C_XLO = 144, C_ACC1 = 288;
constexpr uint32_t C_A2HI = 0, C_A2LO = 64, C_A3HI = 128, C_A3LO = 192, C_RZ = 256, C_GIN = 384, C_GHN = 448;

struct PolParams {
    const float* ring; int64_t n_pad; int64_t n; int32_t slot;       // observation ring, newest slot
    const float* W1rot; const float* Wg; const float* vec;
    const float* hid_in; const uint8_t* reset; float* hid_out;        // [n][NA][64], or env-minor [NA][64][n_pad] (hid_em); reset: h_in = 0 for these envs
    int32_t hid_em;
    float* mean; float* action; float* logp;                          // [n][NA][4]
    const float* eps;                                                 // optional caller-supplied N(0,1) draws [n][NA][4]
    uint64_t seed; uint64_t step; float std_; float log_std; int32_t explore;
    int32_t use_tma;                                                  // observation blocks by one 3-D TMA box copy per tile
    // optional sink for the Transition's `state` (model.py:230-237): the dense get_obs windows [NA][144] of envs [0, st_n) go to
    // rows (st_row0 + e) mod st_cap of pitch st_pitch floats, written by the writer warps from the staged block (TMA path only)
    float* st_out; int64_t st_pitch, st_row0, st_cap, st_n;
};

// One box of the 3-D ring view [24 slots][NA x 6 = agent x feature][n_pad envs], starting at (c_env, c_row, c_slot): box_slots x 6
// x 128 floats -> [6 box_slots][128] in shared memory (k_policy: all 24 slots, k_critic: 12)
__device__ __forceinline__ void tma_load_box(uint32_t dst, const CUtensorMap* map, int32_t c_env, int32_t c_row, int32_t c_slot, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 ::"r"(dst), "l"(map), "r"(c_env), "r"(c_row), "r"(c_slot), "r"(bar) : "memory");
}

constexpr uint32_t IDESC_N64 = umma_idesc_tf32(POL_M, 64), IDESC_N32 = umma_idesc_tf32(POL_M, 32);

__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }

// hi/lo split of four values into the TMEM A operand at columns col (hi part) and col + lo_off (lo part)
__device__ __forceinline__ void split_st4(uint32_t lane_base, uint32_t col_hi, uint32_t col_lo, float a, float b, float c, float d) {
    const float ha = tf32_hi(a), hb = tf32_hi(b), hc = tf32_hi(c), hd = tf32_hi(d);
    tmem_st4(lane_base + col_hi, ha, hb, hc, hd);
    tmem_st4(lane_base + col_lo, __fsub_rn(a, ha), __fsub_rn(b, hb), __fsub_rn(c, hc), __fsub_rn(d, hd));
}

// Gate non-linearities from the SFU exponential (ex2.approx, 2 ulp) and reciprocal: absolute error ~2e-7 on (0, 1) /
// (-1, 1), i.e. fp32 rounding level -- the accurate library tanhf / expf cost 4x the instructions, and the gates are
// 96 evaluations per thread and tile.
// min that propagates a NaN operand (fminf would return the clamp and hide a poisoned row)
__device__ __forceinline__ float min_nan(float a, float b) { float r; asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ float max_nan(float a, float b) { float r; asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ float tanh_fast(float x) {
    const float ax = min_nan(fabsf(x), 15.0f);                       // tanh(15) == 1 in fp32; keeps e^{2x} finite
    const float t = __fsub_rn(1.0f, __fdividef(2.0f, __fadd_rn(__expf(__fmul_rn(2.0f, ax)), 1.0f)));
    return copysignf(t, x);
}

// Four reciprocals from ONE SFU reciprocal: 1 / (a0 a1 a2 a3), multiplied back (9 FMULs).  The GRU cell is SFU-bound (16 lanes
// per clock and SM): its 24 reciprocals per 8 hidden units become 6.  The caller bounds every a_i by 2^29 (clamped gate
// arguments), so the product stays finite; each quotient carries 4 roundings (~2.4e-7 relative at most).
__device__ __forceinline__ float rcp_sfu(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ void rcp4(float a0, float a1, float a2, float a3, float& i0, float& i1, float& i2, float& i3) {
    const float p01 = __fmul_rn(a0, a1), p23 = __fmul_rn(a2, a3);
    const float R = rcp_sfu(__fmul_rn(p01, p23));
    const float r01 = __fmul_rn(R, p23), r23 = __fmul_rn(R, p01);
    i0 = __fmul_rn(r01, a1); i1 = __fmul_rn(r01, a0); i2 = __fmul_rn(r23, a3); i3 = __fmul_rn(r23, a2);
}
// The gate arguments come out of ONE fused multiply-add in the SFU exponential's own unit (base 2): the loader stores the r / z
// biases as -(b_ih + b_hh) log2(e) and the n-gate biases times 2 log2(e) (POL_L2E below).
// 8 sigmoids 1 / (1 + 2^t), t = -(x[i] + b[i]) log2(e) clamped at 20 log2(e) (sigmoid(-20) = 2e-9: below the SFU's error); nb = the stored bias
constexpr float POL_L2E = 1.4426950408889634f;
__device__ __forceinline__ float ex2_sfu(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ void sigmoid8(float (&x)[8], const float* __restrict__ nb) {
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = __fadd_rn(1.0f, ex2_sfu(min_nan(fmaf(x[i], -POL_L2E, nb[i]), 20.0f * POL_L2E)));
    rcp4(x[0], x[1], x[2], x[3], x[0], x[1], x[2], x[3]);
    rcp4(x[4], x[5], x[6], x[7], x[4], x[5], x[6], x[7]);
}
// 8 tanh in place, of u = v / (2 log2(e)): sign(v) (1 - 2 / (2^|v| + 1)), |u| clamped at 10 (tanh(10) == 1 in fp32)
__device__ __forceinline__ void tanh8_scaled(float (&v)[8]) {
    float a[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = __fadd_rn(ex2_sfu(min_nan(fabsf(v[i]), 20.0f * POL_L2E)), 1.0f);
    rcp4(a[0], a[1], a[2], a[3], a[0], a[1], a[2], a[3]);
    rcp4(a[4], a[5], a[6], a[7], a[4], a[5], a[6], a[7]);
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = copysignf(fmaf(-2.0f, a[i], 1.0f), v[i]);
}

// LayerNorm statistics of a row from its four column quarters, CENTRED: a thread reduces its 16 values to (mean_q, M2_q =
// sum of squared deviations from mean_q), and the four pairs merge by Chan's formula, mean = sum mean_q / 4 and
// var = (sum M2_q + 16 sum (mean_q - mean)^2) / 64 (biased, as torch.nn.LayerNorm).  The one-pass SS / 64 - mean^2 loses
// ~(mean / std)^2 ulps of the variance to cancellation, i.e. its error grows with the square of a common offset of the
// pre-activations; centred, only their fp32 representation (~ulp(mean) / std) remains.  A NaN input reaches mean and rstd.
__device__ __forceinline__ float2 ln_quarter(const float (&v)[CPT]) {
    float s = 0.0f;
#pragma unroll
    for (int i = 0; i < CPT; ++i) s = __fadd_rn(s, v[i]);
    const float mq = __fmul_rn(s, 1.0f / CPT);
    float m2 = 0.0f;
#pragma unroll
    for (int i = 0; i < CPT; ++i) { const float d = __fsub_rn(v[i], mq); m2 = fmaf(d, d, m2); }
    return make_float2(mq, m2);
}
// q: the row's first quarter pair, the others POL_M pairs apart; every thread of the row merges them in the same order
__device__ __forceinline__ void ln_merge(const float2* q, float& mean, float& rstd) {
    const float2 t0 = q[0], t1 = q[POL_M], t2 = q[2 * POL_M], t3 = q[3 * POL_M];
    mean = __fmul_rn(__fadd_rn(__fadd_rn(t0.x, t1.x), __fadd_rn(t2.x, t3.x)), 1.0f / TPR);
    const float d0 = __fsub_rn(t0.x, mean), d1 = __fsub_rn(t1.x, mean), d2 = __fsub_rn(t2.x, mean), d3 = __fsub_rn(t3.x, mean);
    const float between = fmaf(d3, d3, fmaf(d2, d2, fmaf(d1, d1, __fmul_rn(d0, d0))));
    const float m2 = __fadd_rn(__fadd_rn(t0.y, t1.y), __fadd_rn(t2.y, t3.y));
    const float var = __fmul_rn(fmaf((float)CPT, between, m2), 1.0f / POL_HID);
    rstd = rsqrtf(__fadd_rn(var, 1e-5f));
}

// the row's four standard normals: the caller's array, or Philox4x32-10 keyed by the seed, counter = (row, step) + Box-Muller.
// They do not depend on the network's output: k_policy draws them while its workers wait for the GRU GEMMs.
__device__ __forceinline__ float4 draw_normals(int64_t r_glob, const float* __restrict__ eps, uint64_t seed, uint64_t step) {
    if (eps != nullptr) return __ldg(reinterpret_cast<const float4*>(eps) + r_glob);
    U4 ctr; ctr.x = (uint32_t)r_glob; ctr.y = (uint32_t)((uint64_t)r_glob >> 32);
    ctr.z = (uint32_t)step; ctr.w = (uint32_t)(step >> 32);
    const U4 rr = philox4x32_10(ctr, (uint32_t)seed, (uint32_t)(seed >> 32));
    // Box-Muller on (0, 1] x [0, 1) uniforms
    const float u0 = ((float)(rr.x >> 8) + 1.0f) * (1.0f / 16777216.0f), u1 = (float)(rr.y >> 8) * (1.0f / 16777216.0f);
    const float u2 = ((float)(rr.z >> 8) + 1.0f) * (1.0f / 16777216.0f), u3 = (float)(rr.w >> 8) * (1.0f / 16777216.0f);
    const float ra = sqrtf(-2.0f * __logf(u0)), rb = sqrtf(-2.0f * __logf(u2));
    float s0, cs0, s1, cs1;
    __sincosf(6.283185307179586f * u1, &s0, &cs0);
    __sincosf(6.283185307179586f * u3, &s1, &cs1);
    return make_float4(ra * cs0, ra * s0, rb * cs1, rb * s1);
}
// explore, given the draw zz: x = m + std z, action = tanh(x), log_prob as above; otherwise status 'test': action = tanh(m)
__device__ __forceinline__ void select_action_drawn(const float (&m)[4], int explore, const float4 zz, float std_, float log_std,
                                                    float (&act)[4], float (&lp)[4]) {
    if (explore) {
        const float z[4] = {zz.x, zz.y, zz.z, zz.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float x = fmaf(std_, z[i], m[i]);              // Normal(mean, std).rsample()
            const float y = tanh_fast(x);
            // Normal.log_prob(x) = -(x - mean)^2 / (2 var) - log(std) - log(sqrt(2 pi)), then the tanh correction
            const float d = __fsub_rn(x, m[i]);
            float l = -__fdividef(__fmul_rn(d, d), __fmul_rn(2.0f, __fmul_rn(std_, std_)));
            l = __fsub_rn(__fsub_rn(l, log_std), 0.9189385332046727f);
            lp[i] = __fsub_rn(l, __logf(__fadd_rn(__fsub_rn(1.0f, __fmul_rn(y, y)), 1e-6f)));
            act[i] = y;
        }
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) { act[i] = tanh_fast(m[i]); lp[i] = 0.0f; }   // status == 'test' (util.py:82-85)
    }
}
__device__ __forceinline__ void select_action_row(const float (&m)[4], int64_t r_glob, int explore, const float* __restrict__ eps,
                                                  uint64_t seed, uint64_t step, float std_, float log_std, float (&act)[4], float (&lp)[4]) {
    const float4 zz = explore ? draw_normals(r_glob, eps, seed, step) : make_float4(0.f, 0.f, 0.f, 0.f);
    select_action_drawn(m, explore, zz, std_, log_std, act, lp);
}

// select_action alone, from stored fc2 outputs (fp_policy_act's d_mean): a second draw for the same policy evaluation --
// train_process evaluates the policy on (next_state, hid) for the next-value action (model.py:225) and AGAIN, on the same
// inputs, at the top of the next step (:215-216); only the exploration draw differs.
__global__ void k_sample(const float* __restrict__ mean, int64_t rows, int explore, const float* __restrict__ eps, uint64_t seed, uint64_t step,
                         float std_, float log_std, float* __restrict__ action, float* __restrict__ logp) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (int64_t)gridDim.x * blockDim.x) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(mean) + r);
        const float m[4] = {t.x, t.y, t.z, t.w};
        float act[4], lp[4];
        select_action_row(m, r, explore, eps, seed, step, std_, log_std, act, lp);
        reinterpret_cast<float4*>(action)[r] = make_float4(act[0], act[1], act[2], act[3]);
        if (logp != nullptr) reinterpret_cast<float4*>(logp)[r] = make_float4(lp[0], lp[1], lp[2], lp[3]);
    }
}

template <int NA>
__global__ void __launch_bounds__(POL_THREADS, 1) k_policy(const PolParams prm, const __grid_constant__ CUtensorMap tmap) {
    extern __shared__ __align__(128) uint8_t smem[];
    const float* vec = reinterpret_cast<const float*>(smem + OFF_VEC);
    float* stage = reinterpret_cast<float*>(smem + OFF_STAGE);
    float2* lnp = reinterpret_cast<float2*>(smem + OFF_LN);
    float4* fcp = reinterpret_cast<float4*>(smem + OFF_FC);
    float4* zdraw = reinterpret_cast<float4*>(smem + OFF_Z);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + OFF_TMEM);
    const uint32_t bar_a = smem_u32(smem + OFF_BAR), bar_m = bar_a + 8, bar_w = bar_a + 16, bar_x = bar_a + 24, bar_q0 = bar_a + 32, bar_s = bar_a + 48;
    const int tid = threadIdx.x, warp = __shfl_sync(0xFFFFFFFFu, tid >> 5, 0);
    const int row = tid & (POL_M - 1), qt = (tid >> 7) & (TPR - 1);        // row of the tile, column quarter
    const bool sink = prm.use_tma && prm.st_out != nullptr;               // the writer warps are at work
    const int64_t n_blocks = (prm.n + POL_M - 1) / POL_M, n_tiles = n_blocks * NA;

    // this tile's observation block: 144 rows (ring slot s, feature f) x 128 envs, each row 512 contiguous bytes.
    // One TMA box copy by the MMA warp (tma_request); rings narrower than a tile take coalesced LDGSTS by the workers.
    auto tma_request = [&](int64_t tile) {                                   // one thread
        mbar_expect_tx(bar_x, POL_OBS * POL_M * 4);
        tma_load_box(smem_u32(stage), &tmap, (int32_t)((tile / NA) * POL_M), (int32_t)(tile % NA) * POL_F, 0, bar_x);
    };
    auto request = [&](int64_t tile) {
        const int a = (int)(tile % NA);
        const int64_t e0 = (tile / NA) * POL_M;
        const int c4 = (tid & 31) * 4;
        const bool inside = e0 + c4 + 4 <= prm.n_pad;
#pragma unroll
        for (int i = 0; i < POL_OBS * 32 / N_WORKERS; ++i) {               // 16-byte chunks: 32 per row, one row per warp and trip
            const int k = (tid >> 5) + (N_WORKERS / 32) * i;
            const int s = k / POL_F, f = k - s * POL_F;
            float* dst = stage + k * POL_M + c4;
            if (inside) cp_async16(dst, prm.ring + ((int64_t)(s * NA + a) * POL_F + f) * prm.n_pad + e0 + c4);
            else *reinterpret_cast<float4*>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        cp_async_commit();
    };

    if (tid == 0) {
        mbar_init(bar_a, N_WORKERS); mbar_init(bar_m, 1); mbar_init(bar_w, 1); mbar_init(bar_x, 1);
        mbar_init(bar_q0, 1); mbar_init(bar_q0 + 8, 1); mbar_init(bar_s, N_WRITERS);
        mbar_init_fence();
        if (prm.use_tma && (int64_t)blockIdx.x < n_tiles) tma_request(blockIdx.x);
        mbar_expect_tx(bar_w, W1_BYTES + WG_BYTES + V_FLOATS * 4);          // weights: three bulk copies, one barrier
        tma_load_1d(smem_u32(smem + OFF_W1), prm.W1rot + (size_t)prm.slot * (W1_BYTES / 4), W1_BYTES, bar_w);
        tma_load_1d(smem_u32(smem + OFF_WG), prm.Wg, WG_BYTES, bar_w);
        tma_load_1d(smem_u32(smem + OFF_VEC), prm.vec, V_FLOATS * 4, bar_w);
    }
    if (warp == 0) {
        tmem_alloc<512>(smem_u32(tmem_slot));
        tmem_relinquish();
    }
    if (!prm.use_tma && tid < N_WORKERS && (int64_t)blockIdx.x < n_tiles) request(blockIdx.x);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == N_WORKERS / 32) {
        // =============================================================== MMA warp
        const uint32_t w1 = smem_u32(smem + OFF_W1), wg = smem_u32(smem + OFF_WG);
        const uint32_t b_rz_ih = wg, b_rz_hh = wg + WG_RZ_BYTES, b_n_ih = wg + 2 * WG_RZ_BYTES, b_n_hh = b_n_ih + WG_N_BYTES;
        uint32_t pa = 0, ps = 0;
        bool first = true;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            // ---- M1: fc1
            mbar_wait(bar_a, pa); pa ^= 1u;
            if (first) { mbar_wait(bar_w, 0u); first = false; }
            tc_fence_after();
            __syncwarp();
            if (elect_one()) {
#pragma unroll
                for (int ks = 0; ks < POL_OBS / 8; ++ks) {
                    const uint64_t db = umma_desc(w1 + ks * 2 * (64 * 16), 64 * 16, 128);
                    umma_tf32_ts(tmem_base + C_ACC1, tmem_base + C_XHI + 8 * ks, db, IDESC_N64, ks > 0 ? 1u : 0u);
                    umma_tf32_ts(tmem_base + C_ACC1, tmem_base + C_XLO + 8 * ks, db, IDESC_N64, 1u);
                }
                umma_commit(bar_m);
            }
            __syncwarp();
            // every worker has read the staging block (P0) -- and, with a `state` sink, so have the writer warps: the next
            // tile's block travels during the GEMM phases.  Requested AFTER fc1's MMAs are on their way: issuing the tensor
            // copy first delayed them -- and with them every worker -- by its issue latency (315 -> 266 us per 131 072 envs)
            if (sink) { mbar_wait(bar_s, ps); ps ^= 1u; }
            if (prm.use_tma && tile + gridDim.x < n_tiles && elect_one()) tma_request(tile + gridDim.x);
            __syncwarp();
            // ---- M2: GRU gates
            mbar_wait(bar_a, pa); pa ^= 1u;
            tc_fence_after();
            __syncwarp();
            if (elect_one()) {
                // The GEMMs are issued in two COLUMN HALVES, each with its own commit: half h holds, for every worker
                // thread of a row, the 8 hidden units of its chunk h (r | z columns adjacent, n-gate blocks alike: the
                // loader permutes the gate rows), i.e. exactly what one trip of the GRU-cell loop below consumes.  The
                // workers start chunk 0 -- bound by the SFUs -- while the tensor pipe still works on half 1, instead of
                // waiting for all the MMAs.  Same MMA cycles (N = 64 / 32 instead of 128 / 64), twice the instructions.
#pragma unroll 1
                for (int hf = 0; hf < 2; ++hf) {
#pragma unroll
                    for (int ks = 0; ks < POL_HID / 8; ++ks) {
                        const uint64_t d_rz_i = umma_desc(b_rz_ih + ks * 2 * (128 * 16) + hf * 64 * 16, 128 * 16, 128);
                        const uint64_t d_rz_h = umma_desc(b_rz_hh + ks * 2 * (128 * 16) + hf * 64 * 16, 128 * 16, 128);
                        const uint64_t d_n_i = umma_desc(b_n_ih + ks * 2 * (64 * 16) + hf * 32 * 16, 64 * 16, 128);
                        const uint64_t d_n_h = umma_desc(b_n_hh + ks * 2 * (64 * 16) + hf * 32 * 16, 64 * 16, 128);
                        umma_tf32_ts(tmem_base + C_RZ + 64 * hf, tmem_base + C_A2HI + 8 * ks, d_rz_i, IDESC_N64, ks > 0 ? 1u : 0u);
                        umma_tf32_ts(tmem_base + C_RZ + 64 * hf, tmem_base + C_A2LO + 8 * ks, d_rz_i, IDESC_N64, 1u);
                        umma_tf32_ts(tmem_base + C_RZ + 64 * hf, tmem_base + C_A3HI + 8 * ks, d_rz_h, IDESC_N64, 1u);
                        umma_tf32_ts(tmem_base + C_RZ + 64 * hf, tmem_base + C_A3LO + 8 * ks, d_rz_h, IDESC_N64, 1u);
                        umma_tf32_ts(tmem_base + C_GIN + 32 * hf, tmem_base + C_A2HI + 8 * ks, d_n_i, IDESC_N32, ks > 0 ? 1u : 0u);
                        umma_tf32_ts(tmem_base + C_GIN + 32 * hf, tmem_base + C_A2LO + 8 * ks, d_n_i, IDESC_N32, 1u);
                        umma_tf32_ts(tmem_base + C_GHN + 32 * hf, tmem_base + C_A3HI + 8 * ks, d_n_h, IDESC_N32, ks > 0 ? 1u : 0u);
                        umma_tf32_ts(tmem_base + C_GHN + 32 * hf, tmem_base + C_A3LO + 8 * ks, d_n_h, IDESC_N32, 1u);
                    }
                    umma_commit(bar_q0 + 8 * hf);
                }
            }
            __syncwarp();
        }
    } else if (warp > N_WORKERS / 32) {
        // =============================================================== writers: the Transition's `state` rows from the staged block
        // A thread owns an env of the tile and walks its 144 window entries (oldest first: ring entry k_out + 6 (slot + 1) mod 144)
        // four at a time: conflict-free shared-memory reads, one 16-byte store per trip into the env's row -- the 32 rows of a
        // warp are 32 different lines, whose sectors the following trips complete while they are still in L2.
        if (sink) {
            const int rot = ((prm.slot + 1) % POL_H) * POL_F;
            uint32_t px = 0;
            for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                const int a = (int)(tile % NA);
                mbar_wait(bar_x, px); px ^= 1u;
                for (int j = tid - (N_WORKERS + 32); j < POL_M; j += N_WRITERS) {      // env of the tile
                    const int64_t e = (tile / NA) * POL_M + j;
                    if (e >= prm.st_n) continue;
                    int64_t orow = prm.st_row0 + e; orow = orow >= prm.st_cap ? orow - prm.st_cap : orow;
                    float4* dst = reinterpret_cast<float4*>(prm.st_out + orow * prm.st_pitch + a * POL_OBS);
#pragma unroll 6
                    for (int kq = 0; kq < POL_OBS / 4; ++kq) {
                        int k = 4 * kq + rot; k = k >= POL_OBS ? k - POL_OBS : k;   // rot and 4 kq are even: k .. k + 3 wrap at most once, never inside a pair
                        const int k2 = (k + 2 >= POL_OBS) ? k + 2 - POL_OBS : k + 2;
                        dst[kq] = make_float4(stage[k * POL_M + j], stage[(k + 1) * POL_M + j], stage[k2 * POL_M + j], stage[(k2 + 1) * POL_M + j]);
                    }
                }
                mbar_arrive(bar_s);
            }
        }
    } else {
        // =============================================================== workers: four threads per row (column quarters)
        const uint32_t lane_base = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
        const int c0 = CPT * qt;                                               // this thread's 16 hidden columns
        uint32_t pm = 0, px = 0, pq = 0;
        bool first = true;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const int a = (int)(tile % NA);
            const int64_t e = (tile / NA) * POL_M + row;
            const bool live = e < prm.n;
            const int64_t r_glob = e * NA + a;                                  // row of the reference's (b, n, .) tensors

            // ---- P0: observation block -> TMEM (this thread: 36 of the row's 144 inputs)
            if (prm.use_tma) { mbar_wait(bar_x, px); px ^= 1u; }
            else cp_async_wait_all();
            group_sync<1, N_WORKERS>();                                         // the block has landed; TMEM of the previous tile is drained
#pragma unroll
            for (int c = 0; c < KPT / 4; ++c) {
                const int k0 = KPT * qt + 4 * c;
                split_st4(lane_base, C_XHI + k0, C_XLO + k0, stage[(k0 + 0) * POL_M + row], stage[(k0 + 1) * POL_M + row],
                          stage[(k0 + 2) * POL_M + row], stage[(k0 + 3) * POL_M + row]);
            }
            tmem_wait_st();
            tc_fence_before();
            mbar_arrive(bar_a);
            if (!prm.use_tma) {
                group_sync<1, N_WORKERS>();                                     // every thread has read the staging block
                if (tile + gridDim.x < n_tiles) request(tile + gridDim.x);
            }
            // the previous hidden state of this thread's 16 units (issued now, consumed after fc1)
            float h[CPT];
            {
                const bool zero = !live || prm.hid_in == nullptr || (prm.reset != nullptr && prm.reset[e] != 0);
                if (prm.hid_em) {                                               // env-minor: one coalesced 128-byte line per unit and warp
                    const float* hp = prm.hid_in + (zero ? 0 : ((int64_t)(a * POL_HID + c0) * prm.n_pad + e));
#pragma unroll
                    for (int i = 0; i < CPT; ++i) h[i] = zero ? 0.0f : __ldg(hp + (int64_t)i * prm.n_pad);
                } else {
                    const float4* hp = reinterpret_cast<const float4*>(prm.hid_in + (zero ? 0 : r_glob) * POL_HID + c0);
#pragma unroll
                    for (int i = 0; i < CPT / 4; ++i) {
                        const float4 t = zero ? make_float4(0.f, 0.f, 0.f, 0.f) : __ldg(hp + i);
                        h[4 * i] = t.x; h[4 * i + 1] = t.y; h[4 * i + 2] = t.z; h[4 * i + 3] = t.w;
                    }
                }
            }
            if (first) { mbar_wait(bar_w, 0u); first = false; }                 // the small arrays have landed

            // ---- E1: fc1 epilogue: bias(agent), LayerNorm, ReLU -> A2; h -> A3
            mbar_wait(bar_m, pm); pm ^= 1u;
            tc_fence_after();
            {
                float v[CPT];
                tmem_ld16(lane_base + C_ACC1 + c0, v);
                tmem_wait_ld();
#pragma unroll
                for (int i = 0; i < CPT; ++i) v[i] = __fadd_rn(v[i], vec[V_B1A + a * POL_HID + c0 + i]);
                lnp[qt * POL_M + row] = ln_quarter(v);
                group_sync<1, N_WORKERS>();
                float mean, rstd;
                ln_merge(lnp + row, mean, rstd);
#pragma unroll
                for (int i = 0; i < CPT; ++i) {
                    const float y = fmaf(__fmul_rn(__fsub_rn(v[i], mean), rstd), vec[V_LNG + c0 + i], vec[V_LNB + c0 + i]);
                    v[i] = max_nan(y, 0.0f);                                      // hid_activation = relu
                }
#pragma unroll
                for (int c = 0; c < CPT / 4; ++c) {
                    split_st4(lane_base, C_A2HI + c0 + 4 * c, C_A2LO + c0 + 4 * c, v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
                    split_st4(lane_base, C_A3HI + c0 + 4 * c, C_A3LO + c0 + 4 * c, h[4 * c], h[4 * c + 1], h[4 * c + 2], h[4 * c + 3]);
                }
            }
            tmem_wait_st();
            tc_fence_before();
            mbar_arrive(bar_a);
            // the exploration draw of this row (Philox + Box-Muller: ~140 dependent instructions of the sampling thread) does not
            // depend on the network: drawn here, while the tensor pipe works on the GRU GEMMs, kept in shared memory (same thread)
            if (qt == 0 && live && prm.explore) zdraw[row] = draw_normals(r_glob, prm.eps, prm.seed, prm.step);

            // ---- E2: GRU cell (torch.nn.GRUCell: r, z, n gate order) -> h'; fc2 partial sums
            {
                float p0 = 0.0f, p1 = 0.0f, p2 = 0.0f, p3 = 0.0f;
#pragma unroll
                for (int hc = 0; hc < CPT / 8; ++hc) {                          // two chunks of 8 columns: half the live registers
                    const int cc = c0 + 8 * hc;
                    float rp[8], zp[8], gi[8], gh[8];
                    mbar_wait(bar_q0 + 8 * hc, pq);                             // column half hc of the GRU GEMMs: [quarter][r8 | z8], [quarter][n8]
                    tc_fence_after();
                    tmem_ld8(lane_base + C_RZ + 64 * hc + 16 * qt, rp);
                    tmem_ld8(lane_base + C_RZ + 64 * hc + 16 * qt + 8, zp);
                    tmem_ld8(lane_base + C_GIN + 32 * hc + 8 * qt, gi);
                    tmem_ld8(lane_base + C_GHN + 32 * hc + 8 * qt, gh);
                    tmem_wait_ld();
                    sigmoid8(rp, vec + V_BRZ + cc);                             // r
                    sigmoid8(zp, vec + V_BRZ + 64 + cc);                        // z
#pragma unroll
                    for (int i = 0; i < 8; ++i)                                 // 2 log2(e) (gi_n + b_in + r (gh_n + b_hn))
                        gi[i] = fmaf(rp[i], fmaf(gh[i], 2.0f * POL_L2E, vec[V_BHN + cc + i]), fmaf(gi[i], 2.0f * POL_L2E, vec[V_BIN + cc + i]));
                    tanh8_scaled(gi);                                           // n = tanh(gi_n + r gh_n)
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float z = zp[i], nn = gi[i];
                        const float hn = fmaf(z, __fsub_rn(h[8 * hc + i], nn), nn);   // (1 - z) n + z h
                        h[8 * hc + i] = hn;
                        const float4 w2 = *reinterpret_cast<const float4*>(vec + V_W2 + 4 * (cc + i));   // fc2's column of unit cc + i: one LDS.128
                        p0 = fmaf(hn, w2.x, p0); p1 = fmaf(hn, w2.y, p1); p2 = fmaf(hn, w2.z, p2); p3 = fmaf(hn, w2.w, p3);
                    }
                }
                pq ^= 1u;
                fcp[qt * POL_M + row] = make_float4(p0, p1, p2, p3);
                if (live && prm.hid_em) {
                    float* ho = prm.hid_out + (int64_t)(a * POL_HID + c0) * prm.n_pad + e;
#pragma unroll
                    for (int i = 0; i < CPT; ++i) ho[(int64_t)i * prm.n_pad] = h[i];
                } else if (live) {
                    float4* ho = reinterpret_cast<float4*>(prm.hid_out + r_glob * POL_HID + c0);
#pragma unroll
                    for (int i = 0; i < CPT / 4; ++i) ho[i] = make_float4(h[4 * i], h[4 * i + 1], h[4 * i + 2], h[4 * i + 3]);
                }
            }
            tc_fence_before();
            group_sync<1, N_WORKERS>();                                         // the partial sums of the row are in place

            // ---- fc2 bias + select_action (utils/util.py:50-64)
            if (qt == 0 && live) {
                float m[4];
                {
                    const float4 t0 = fcp[row], t1 = fcp[POL_M + row], t2 = fcp[2 * POL_M + row], t3 = fcp[3 * POL_M + row];
                    m[0] = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(t0.x, t1.x), t2.x), t3.x), vec[V_B2 + 0]);
                    m[1] = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(t0.y, t1.y), t2.y), t3.y), vec[V_B2 + 1]);
                    m[2] = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(t0.z, t1.z), t2.z), t3.z), vec[V_B2 + 2]);
                    m[3] = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(t0.w, t1.w), t2.w), t3.w), vec[V_B2 + 3]);
                }
                if (prm.mean != nullptr) reinterpret_cast<float4*>(prm.mean)[r_glob] = make_float4(m[0], m[1], m[2], m[3]);
                float act[4], lp[4];
                select_action_drawn(m, prm.explore, zdraw[row], prm.std_, prm.log_std, act, lp);
                reinterpret_cast<float4*>(prm.action)[r_glob] = make_float4(act[0], act[1], act[2], act[3]);
                if (prm.logp != nullptr) reinterpret_cast<float4*>(prm.logp)[r_glob] = make_float4(lp[0], lp[1], lp[2], lp[3]);
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<512>(tmem_base);
}

// ---------------------------------------------------------------------------- critic: MADDPG.value on tcgen05
// k_critic replaces, for N envs x NA agents at once, MADDPG.value (madrl/models/maddpg.py:29-76) with the shared-parameter
// MLPCritic (madrl/critics/mlp_critic.py:5-36: fc1 -> LayerNorm -> ReLU -> fc2 -> ReLU -> fc3) as train_process calls it for
// the Transition's value / next_value (madrl/models/model.py:217, :225-226).  The critic's 149 NA-wide input row of (env,
// agent i) is [all agents' observations (144 NA) | one-hot(i) (NA) | all agents' actions (4 NA)] (745 for five agents):
// only the one-hot differs between the NA rows of an env, so fc1 is evaluated ONCE per env on its 148 NA shared columns and the one-hot column is
// folded into a per-agent bias.  A tile is 128 envs, input = the env-minor observation ring, untouched:
//   fc1: 2 NA HALF-BLOCKS per tile (agent a, ring slots 12 hf .. 12 hf + 11: K = 72).  A half-block is one TMA box [12][6][128]
//        into one of three staging buffers (requested three half-blocks ahead: the HBM stream never waits for the workers)
//        plus the matching half of agent a's fc1 block -- ring rotation folded into the weights like k_policy's W1 -- into
//        one of four weight buffers (two ahead); the workers split it into one of two TMEM operand buffers while the MMAs
//        of the previous half-block run (acc1 += X Wc^T: 9 k-steps x (hi, lo)); the first half-block also adds the actions'
//        4 NA columns (K padded to 24)
//   per agent i = 0 .. NA - 1: E1: acc1 + bias(i) -> LayerNorm -> ReLU -> split -> A2[i & 1];  M2: acc2[i & 1] = A2 W2^T;  E2: ReLU,
//        dot with fc3 (fp32, CUDA cores), four-thread reduction, + bias -> value[env][i];  operand and accumulator are
//        double-buffered: E1 of agent i + 1 runs under fc2 of agent i
// Workers and the MMA warp meet through two mbarrier pairs (a_ready[b], mma_done[b], b = TMEM buffer); every commit is
// awaited exactly once per worker, in order.  Precision as k_policy: activations two-term TF32 split, fc1 / fc2 matrices
// held as TF32, fc3 in fp32.
constexpr int CR_KH = POL_OBS / 2;                                           // K of a half-block: 72
constexpr int CR_NST = 3, CR_NWB = 4;                                        // staging buffers, weight buffers in flight
constexpr uint32_t CR_ST_BYTES = CR_KH * POL_M * 4;                          // [72][128] fp32 = 36 864
constexpr uint32_t CR_WB_BYTES = W1_BYTES;                                   // one agent block of fc1: [36 kc][64 n][4]
constexpr uint32_t CR_WH_BYTES = CR_WB_BYTES / 2;                            // ... and its half: [18 kc][64 n][4] = 18 432
constexpr uint32_t CR_W2_BYTES = POL_HID * POL_HID * 4;                      // fc2: [16 kc][64 n][4]
constexpr int CR_KACT = 24;                                                  // 20 action columns + 4 zero columns
constexpr uint32_t CR_WA_BYTES = CR_KACT * POL_HID * 4;                      // [6 kc][64 n][4]
// small arrays (floats): b1a[5][64] (fc1.bias + the one-hot column of agent i), ln_g[64], ln_b[64], b2[64], w3[64], b3 (+ pad)
constexpr int CV_B1A = 0, CV_LNG = 320, CV_LNB = 384, CV_B2 = 448, CV_W3 = 512, CV_B3 = 576, CV_FLOATS = 592;
constexpr uint32_t CO_ST = 0, CO_WB = CO_ST + CR_NST * CR_ST_BYTES, CO_W2 = CO_WB + CR_NWB * CR_WH_BYTES, CO_WA = CO_W2 + CR_W2_BYTES,
                   CO_VEC = CO_WA + CR_WA_BYTES;
constexpr uint32_t CO_LN = (CO_VEC + CV_FLOATS * 4 + 127) / 128 * 128;       // [2][TPR][128 rows] float2
constexpr uint32_t CO_FC = CO_LN + 2 * TPR * POL_M * 8;                      // [2][TPR][128 rows] float: fc3 partial sums
constexpr uint32_t CO_BAR = CO_FC + 2 * TPR * POL_M * 4;                     // a_ready[2], mma_done[2], small arrays, x_full[3], wb[4]
constexpr uint32_t CO_TMEM = CO_BAR + 96;
constexpr uint32_t CR_SMEM = CO_TMEM + 16;
static_assert(CR_SMEM <= 227 * 1024, "critic kernel exceeds the shared memory of one SM");
static_assert(CO_WB % 128 == 0 && CO_W2 % 128 == 0 && CO_WA % 128 == 0 && CO_VEC % 16 == 0 && CO_BAR % 8 == 0, "operand alignment");
// TMEM columns: operand buffer b at 144 b: hi [0, 72) | lo [72, 144) (fc2's operands A2[0] / A2[1] alias the buffers: hi at
// +0, lo at +64), acc1, acc2[0], acc2[1] (the actions' operand of the first half-block aliases acc2[1])
constexpr uint32_t CC_XB = 2 * CR_KH, CC_ACC1 = 288, CC_ACC2_0 = 352, CC_ACC2_1 = 416, CC_ACTHI = 416, CC_ACTLO = 440;
static_assert(2 * CC_XB == CC_ACC1 && CC_XB + 128 <= CC_ACC1 && CC_ACC2_1 + 64 <= 512, "TMEM map");

struct CritParams {
    const float* ring; int64_t n_pad; int64_t n; int32_t slot;
    const float* Wc1rot; const float* W2; const float* Wa; const float* vec;
    const float* actions;                                             // [n][NA][4]
    float* value;                                                     // [n][NA]
    int32_t use_tma;
};

template <int NA>
__global__ void __launch_bounds__(CRIT_THREADS, 1) k_critic(const CritParams prm, const __grid_constant__ CUtensorMap tmap) {
    constexpr int CR_HB = 2 * NA;                                            // half-blocks per tile
    extern __shared__ __align__(128) uint8_t smem[];
    const float* vec = reinterpret_cast<const float*>(smem + CO_VEC);
    float2* lnp = reinterpret_cast<float2*>(smem + CO_LN);
    float* fcp = reinterpret_cast<float*>(smem + CO_FC);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + CO_TMEM);
    const uint32_t bar_a0 = smem_u32(smem + CO_BAR), bar_m0 = bar_a0 + 16, bar_w = bar_a0 + 32, bar_x0 = bar_a0 + 40, bar_wb0 = bar_a0 + 64;
    const int tid = threadIdx.x, warp = __shfl_sync(0xFFFFFFFFu, tid >> 5, 0);
    const int row = tid & (POL_M - 1), qt = (tid >> 7) & (TPR - 1);
    const int64_t n_tiles = (prm.n + POL_M - 1) / POL_M;
    const int64_t n_my = (n_tiles > (int64_t)blockIdx.x) ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int64_t n_hb = n_my * CR_HB;                                       // half-blocks of this CTA, in order: g = 2 NA tile + 2 a + hf

    auto tile_of = [&](int64_t g) -> int64_t { return (int64_t)blockIdx.x + (g / CR_HB) * gridDim.x; };
    auto tma_request = [&](int64_t g) {                                      // one thread: half-block g -> staging buffer g % 3
        const uint32_t bar = bar_x0 + 8 * (uint32_t)(g % CR_NST);
        const int a = (int)((g % CR_HB) >> 1), hf = (int)(g & 1);
        mbar_expect_tx(bar, CR_ST_BYTES);
        tma_load_box(smem_u32(smem + CO_ST + (g % CR_NST) * CR_ST_BYTES), &tmap, (int32_t)(tile_of(g) * POL_M), a * POL_F,
                     hf * (POL_H / 2), bar);
    };
    auto load_wb = [&](int64_t g) {                                          // one thread: fc1 half-block weights -> buffer g % 4
        const uint32_t bar = bar_wb0 + 8 * (uint32_t)(g % CR_NWB);
        const size_t a = (size_t)((g % CR_HB) >> 1), hf = (size_t)(g & 1);
        mbar_expect_tx(bar, CR_WH_BYTES);
        tma_load_1d(smem_u32(smem + CO_WB + (g % CR_NWB) * CR_WH_BYTES),
                    prm.Wc1rot + (((size_t)prm.slot * NA + a) * 2 + hf) * (CR_WH_BYTES / 4), CR_WH_BYTES, bar);
    };
    auto request = [&](int64_t g) {                                          // workers, rings narrower than a tile: LDGSTS, not pipelined
        const int a = (int)((g % CR_HB) >> 1), hf = (int)(g & 1);
        const int64_t e0 = tile_of(g) * POL_M;
        float* stage = reinterpret_cast<float*>(smem + CO_ST + (g % CR_NST) * CR_ST_BYTES);
        const int c4 = (tid & 31) * 4;
        const bool inside = e0 + c4 + 4 <= prm.n_pad;
        for (int k = tid >> 5; k < CR_KH; k += N_WORKERS / 32) {              // 16-byte chunks: 32 per row, one row per warp and trip
            const int sl = hf * (POL_H / 2) + k / POL_F, f = k % POL_F;
            float* dst = stage + k * POL_M + c4;
            if (inside) cp_async16(dst, prm.ring + ((int64_t)(sl * NA + a) * POL_F + f) * prm.n_pad + e0 + c4);
            else *reinterpret_cast<float4*>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        cp_async_commit();
    };

    if (tid == 0) {
        mbar_init(bar_a0, N_WORKERS); mbar_init(bar_a0 + 8, N_WORKERS); mbar_init(bar_m0, 1); mbar_init(bar_m0 + 8, 1);
        mbar_init(bar_w, 1);
        for (int i = 0; i < CR_NST; ++i) mbar_init(bar_x0 + 8 * i, 1);
        for (int i = 0; i < CR_NWB; ++i) mbar_init(bar_wb0 + 8 * i, 1);
        mbar_init_fence();
        for (int64_t g = 0; g < CR_NST && g < n_hb; ++g) if (prm.use_tma) tma_request(g);
        for (int64_t g = 0; g < 2 && g < n_hb; ++g) load_wb(g);
        mbar_expect_tx(bar_w, CR_W2_BYTES + CR_WA_BYTES + CV_FLOATS * 4);    // fc2, action columns, small arrays: one barrier
        tma_load_1d(smem_u32(smem + CO_W2), prm.W2, CR_W2_BYTES, bar_w);
        tma_load_1d(smem_u32(smem + CO_WA), prm.Wa, CR_WA_BYTES, bar_w);
        tma_load_1d(smem_u32(smem + CO_VEC), prm.vec, CV_FLOATS * 4, bar_w);
    }
    if (warp == 0) {
        tmem_alloc<512>(smem_u32(tmem_slot));
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == N_WORKERS / 32) {
        // =============================================================== MMA warp
        const uint32_t w2 = smem_u32(smem + CO_W2), wa = smem_u32(smem + CO_WA);
        uint32_t pa0 = 0u, pa1 = 0u;                                        // phase parities of a_ready[0] / [1]
        bool first = true;
        for (int64_t g = 0; g < n_hb; ++g) {
            const int hb = (int)(g % CR_HB), b = (int)(g & 1);
            // ---- fc1, half-block g (K = 72; the tile's first one: + the actions)
            if (b) { mbar_wait(bar_a0 + 8, pa1); pa1 ^= 1u; } else { mbar_wait(bar_a0, pa0); pa0 ^= 1u; }
            mbar_wait(bar_wb0 + 8 * (uint32_t)(g % CR_NWB), (uint32_t)((g / CR_NWB) & 1));
            if (first) { mbar_wait(bar_w, 0u); first = false; }
            tc_fence_after();
            __syncwarp();
            if (elect_one()) {
                const uint32_t wb = smem_u32(smem + CO_WB + (g % CR_NWB) * CR_WH_BYTES), xb = tmem_base + CC_XB * b;
                // one descriptor per half-block: a k-step advances its 16-byte-granular start address by a constant (the address
                // field cannot carry: shared memory ends far below 2^18)
                const uint64_t d0 = umma_desc(wb, 64 * 16, 128);
#pragma unroll
                for (int ks = 0; ks < CR_KH / 8; ++ks) {
                    const uint64_t db = d0 + (uint64_t)((ks * 2 * (64 * 16)) >> 4);
                    umma_tf32_ts(tmem_base + CC_ACC1, xb + 8 * ks, db, IDESC_N64, (hb > 0 || ks > 0) ? 1u : 0u);
                    umma_tf32_ts(tmem_base + CC_ACC1, xb + CR_KH + 8 * ks, db, IDESC_N64, 1u);
                }
                if (hb == 0) {
#pragma unroll
                    for (int ks = 0; ks < CR_KACT / 8; ++ks) {
                        const uint64_t db = umma_desc(wa + ks * 2 * (64 * 16), 64 * 16, 128);
                        umma_tf32_ts(tmem_base + CC_ACC1, tmem_base + CC_ACTHI + 8 * ks, db, IDESC_N64, 1u);
                        umma_tf32_ts(tmem_base + CC_ACC1, tmem_base + CC_ACTLO + 8 * ks, db, IDESC_N64, 1u);
                    }
                }
                umma_commit(bar_m0 + 8 * b);
                // every worker has read staging buffer g % 3, and the MMAs of half-block g - 2 have completed (the workers waited
                // for them before writing this operand buffer): half-block g + 3 and the weights of g + 2 may travel -- requested
                // AFTER the MMAs are on their way (issuing the copies first delays them by the copies' issue latency)
                if (prm.use_tma && g + CR_NST < n_hb) tma_request(g + CR_NST);
                if (g + 2 < n_hb) load_wb(g + 2);
            }
            __syncwarp();
            if (hb != CR_HB - 1) continue;
            // ---- fc2, once per agent row, operand / accumulator buffer i & 1
            for (int i = 0; i < NA; ++i) {
                const int bi = i & 1;
                if (bi) { mbar_wait(bar_a0 + 8, pa1); pa1 ^= 1u; } else { mbar_wait(bar_a0, pa0); pa0 ^= 1u; }
                tc_fence_after();
                __syncwarp();
                if (elect_one()) {
                    const uint32_t a2 = tmem_base + CC_XB * bi, acc = tmem_base + (bi ? CC_ACC2_1 : CC_ACC2_0);
#pragma unroll
                    for (int ks = 0; ks < POL_HID / 8; ++ks) {
                        const uint64_t db = umma_desc(w2 + ks * 2 * (64 * 16), 64 * 16, 128);
                        umma_tf32_ts(acc, a2 + 8 * ks, db, IDESC_N64, ks > 0 ? 1u : 0u);
                        umma_tf32_ts(acc, a2 + 64 + 8 * ks, db, IDESC_N64, 1u);
                    }
                    umma_commit(bar_m0 + 8 * bi);
                }
                __syncwarp();
            }
        }
    } else if (warp < N_WORKERS / 32) {
        // =============================================================== workers: four threads per env row (column quarters)
        const uint32_t lane_base = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
        const int c0 = CPT * qt;
        uint32_t pm0 = 0u, pm1 = 0u;                                            // phase parities of mma_done[0] / [1]
        bool first = true;
        for (int64_t g = 0; g < n_hb; ++g) {
            const int hb = (int)(g % CR_HB), b = (int)(g & 1);
            const int64_t e = tile_of(g) * POL_M + row;
            const bool live = e < prm.n;
            const float* stage = reinterpret_cast<const float*>(smem + CO_ST + (g % CR_NST) * CR_ST_BYTES);
            // ---- P0: half-block g -> TMEM operand buffer b
            if (prm.use_tma) mbar_wait(bar_x0 + 8 * (uint32_t)(g % CR_NST), (uint32_t)((g / CR_NST) & 1));
            else { request(g); cp_async_wait_all(); group_sync<1, N_WORKERS>(); }
            if (hb >= 2) { if (b) { mbar_wait(bar_m0 + 8, pm1); pm1 ^= 1u; } else { mbar_wait(bar_m0, pm0); pm0 ^= 1u; } tc_fence_after(); }   // the MMAs of half-block g - 2 have read this buffer
            const uint32_t xhi = CC_XB * b, xlo = xhi + CR_KH;
#pragma unroll
            for (int c = 0; c < 4; ++c) {                                       // K [0, 64): chunks of 16, four per thread
                const int k0 = 16 * c + 4 * qt;
                split_st4(lane_base, xhi + k0, xlo + k0, stage[(k0 + 0) * POL_M + row], stage[(k0 + 1) * POL_M + row],
                          stage[(k0 + 2) * POL_M + row], stage[(k0 + 3) * POL_M + row]);
            }
            if (qt < 2) {                                                       // K [64, 72)
                const int k0 = 64 + 4 * qt;
                split_st4(lane_base, xhi + k0, xlo + k0, stage[(k0 + 0) * POL_M + row], stage[(k0 + 1) * POL_M + row],
                          stage[(k0 + 2) * POL_M + row], stage[(k0 + 3) * POL_M + row]);
            }
            if (hb == 0 && qt < 3) {                                            // the env's 4 NA action values (+ zero columns to 24): 8 per thread
                float v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int k = 8 * qt + i;
                    v[i] = (live && k < NA * POL_ACT) ? __ldg(prm.actions + e * (NA * POL_ACT) + k) : 0.0f;
                }
                split_st4(lane_base, CC_ACTHI + 8 * qt, CC_ACTLO + 8 * qt, v[0], v[1], v[2], v[3]);
                split_st4(lane_base, CC_ACTHI + 8 * qt + 4, CC_ACTLO + 8 * qt + 4, v[4], v[5], v[6], v[7]);
            }
            tmem_wait_st();
            tc_fence_before();
            mbar_arrive(bar_a0 + 8 * b);
            if (!prm.use_tma) group_sync<1, N_WORKERS>();                       // every thread has read the staging buffer (LDGSTS path refills it)
            if (hb != CR_HB - 1) continue;

            // ---- per agent row: E1 (bias, LayerNorm, ReLU -> A2[i & 1]) | fc2 | E2 (ReLU, fc3); E1 of agent i + 1 runs under fc2 of agent i
            if (first) { mbar_wait(bar_w, 0u); first = false; }                 // the small arrays have landed
            mbar_wait(bar_m0, pm0); pm0 ^= 1u;                              // fc1 is complete: the tile's last two half-blocks
            mbar_wait(bar_m0 + 8, pm1); pm1 ^= 1u;
            tc_fence_after();
            float y1[CPT];
            tmem_ld16(lane_base + CC_ACC1 + c0, y1);
            tmem_wait_ld();
            auto e1 = [&](int i) {
                float v[CPT];
#pragma unroll
                for (int c = 0; c < CPT; ++c) v[c] = __fadd_rn(y1[c], vec[CV_B1A + i * POL_HID + c0 + c]);
                float2* ln = lnp + (i & 1) * (TPR * POL_M);
                ln[qt * POL_M + row] = ln_quarter(v);
                group_sync<1, N_WORKERS>();
                float mean, rstd;
                ln_merge(ln + row, mean, rstd);
#pragma unroll
                for (int c = 0; c < CPT; ++c) {
                    const float t = fmaf(__fmul_rn(__fsub_rn(v[c], mean), rstd), vec[CV_LNG + c0 + c], vec[CV_LNB + c0 + c]);
                    v[c] = max_nan(t, 0.0f);                                      // hid_activation = relu
                }
                const uint32_t a2 = CC_XB * (i & 1);
#pragma unroll
                for (int c = 0; c < CPT / 4; ++c)
                    split_st4(lane_base, a2 + c0 + 4 * c, a2 + 64 + c0 + 4 * c, v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
                tmem_wait_st();
                tc_fence_before();
                mbar_arrive(bar_a0 + 8 * (i & 1));
            };
            e1(0);
            for (int i = 0; i < NA; ++i) {
                const int bi = i & 1;
                if (i + 1 < NA) e1(i + 1);                                  // (its operand buffer was released by E2 of agent i - 1)
                if (bi) { mbar_wait(bar_m0 + 8, pm1); pm1 ^= 1u; } else { mbar_wait(bar_m0, pm0); pm0 ^= 1u; }
                tc_fence_after();
                float u[CPT];
                tmem_ld16(lane_base + (bi ? CC_ACC2_1 : CC_ACC2_0) + c0, u);
                tmem_wait_ld();
                float part = 0.0f;
#pragma unroll
                for (int c = 0; c < CPT; ++c) part = fmaf(max_nan(__fadd_rn(u[c], vec[CV_B2 + c0 + c]), 0.0f), vec[CV_W3 + c0 + c], part);
                float* fc = fcp + bi * (TPR * POL_M);
                fc[qt * POL_M + row] = part;
                tc_fence_before();
                group_sync<1, N_WORKERS>();
                if (qt == 0 && live)
                    prm.value[e * NA + i] = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(fc[row], fc[POL_M + row]), fc[2 * POL_M + row]), fc[3 * POL_M + row]), vec[CV_B3]);
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<512>(tmem_base);
}

// ---------------------------------------------------------------------------- transitions -> replay ring, learner feed
// Pure data movement.  The sources are env-minor ([row][n_pad]: the observation ring, the hidden states), the replay
// fields env-major ([transition][width]): a transposition through shared memory in tiles of GT_ENVS = 128 envs, so that
// both sides move >= 512 contiguous bytes per row (a 32-env tile reads 128-byte pieces 512 KB apart: 2.8 TB/s; this one
// reads 512-byte pieces).  Tile [KR rows][129] floats (odd stride: both the row-wise fill and the column-wise drain are
// conflict-free); the fill issues all of a thread's loads before the first store.
constexpr int GT_ENVS = 128, GT_STRIDE = GT_ENVS + 1;

template <int KR, class RowOf>
__device__ __forceinline__ void gt_fill(float* t, const float* __restrict__ src, int64_t n_pad, int64_t e0, int64_t n, RowOf row_of,
                                        const uint8_t* __restrict__ zero_mask) {
    static_assert(KR % 16 == 0, "rows per tile: two batches of KR / 16 rows per warp");
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    bool take[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int64_t e = e0 + lane + 32 * i;
        take[i] = (e < n) && (zero_mask == nullptr || zero_mask[e] == 0);
    }
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        float v[KR / 16][4];
#pragma unroll
        for (int m = 0; m < KR / 16; ++m) {
            const int k = w + 8 * (m + half * (KR / 16));
            const float* sp = src + (int64_t)row_of(k) * n_pad + e0 + lane;
#pragma unroll
            for (int i = 0; i < 4; ++i) v[m][i] = take[i] ? __ldg(sp + 32 * i) : 0.0f;
        }
#pragma unroll
        for (int m = 0; m < KR / 16; ++m) {
            const int k = w + 8 * (m + half * (KR / 16));
#pragma unroll
            for (int i = 0; i < 4; ++i) t[k * GT_STRIDE + lane + 32 * i] = v[m][i];
        }
    }
}
// rows (row0 + e) mod cap of the field, columns [col0, col0 + KR) of a row of `pitch` floats
template <int KR>
__device__ __forceinline__ void gt_drain(const float* t, float* __restrict__ out, int64_t pitch, int col0, int64_t e0, int64_t n,
                                         int64_t row0, int64_t cap) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll 4
    for (int j = w; j < GT_ENVS; j += 8) {
        if (e0 + j < n) {
            int64_t orow = row0 + e0 + j; orow = orow >= cap ? orow - cap : orow;
            float* dst = out + orow * pitch + col0;
#pragma unroll
            for (int k = lane; k < KR; k += 32) dst[k] = t[k * GT_STRIDE + j];
        }
    }
}

//   k_window_gather   dense observation windows [n][NA][144] (oldest entry first: get_obs, :387-401) of envs [0, n) from
//                     the env-minor ring into rows of pitch `pitch` floats (a replay field, or a dense tensor)
template <int NA>
__global__ void __launch_bounds__(256) k_window_gather(const float* __restrict__ ring, int64_t n_pad, int slot, int64_t n,
                                                       float* __restrict__ out, int64_t pitch, int64_t row0, int64_t cap) {
    extern __shared__ float gt_tile[];                            // [144][129]
    const int64_t n_blk = (n + GT_ENVS - 1) / GT_ENVS;
    for (int64_t blk = blockIdx.x; blk < n_blk * NA; blk += gridDim.x) {
        const int a = (int)(blk % NA);
        const int64_t e0 = (blk / NA) * GT_ENVS;
        // k = r * 6 + f: the r-th oldest entry lives in ring slot (slot + 1 + r) mod 24
        gt_fill<POL_OBS>(gt_tile, ring, n_pad, e0, n, [&](int k) {
            const int r = k / POL_F, f = k - r * POL_F;
            int s = slot + 1 + r; s = s >= POL_H ? s - POL_H : s;
            return (s * NA + a) * POL_F + f;
        }, nullptr);
        __syncthreads();
        gt_drain<POL_OBS>(gt_tile, out, pitch, a * POL_OBS, e0, n, row0, cap);
        __syncthreads();
    }
}

// env-minor [NA x 64 units][n_pad] -> ring rows (row0 + e) mod cap of NA x 64 contiguous floats: the hidden states of the
// Transition (last_hid / hid, (1, NA, 64) per env) from the policy kernel's native layout; a tile is (128 envs, one half
// of the NA x 64 rows)
template <int NA>
__global__ void __launch_bounds__(256) k_em_gather(const float* __restrict__ src, int64_t n_pad, int64_t n,
                                                   float* __restrict__ out, int64_t row0, int64_t cap,
                                                   const uint8_t* __restrict__ zero_mask) {
    constexpr int EM_ROWS = NA * POL_HID, EM_KR = EM_ROWS / 2;
    extern __shared__ float gt_tile[];                            // [EM_KR][129]
    const int64_t n_blk = (n + GT_ENVS - 1) / GT_ENVS;
    for (int64_t blk = blockIdx.x; blk < n_blk * 2; blk += gridDim.x) {
        const int h = (int)(blk & 1);
        const int64_t e0 = (blk >> 1) * GT_ENVS;
        gt_fill<EM_KR>(gt_tile, src, n_pad, e0, n, [&](int k) { return h * EM_KR + k; }, zero_mask);
        __syncthreads();
        gt_drain<EM_KR>(gt_tile, out, EM_ROWS, h * EM_KR, e0, n, row0, cap);
        __syncthreads();
    }
}

// rows of `width` floats from a dense [n][width] source into ring rows (row0 + e) mod cap of pitch `width`
__global__ void k_rows_to_ring(const float* __restrict__ src, int64_t n, int width, float* __restrict__ dst, int64_t row0, int64_t cap) {
    const int64_t total = n * width, ring = cap * width, base = row0 * width;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t o = base + i; o = o >= ring ? o - ring : o;
        dst[o] = src[i];
    }
}

// reward (fp64, one per env) repeated for the agents (model.py:221), done / last_step flags, all-ones availability
template <int NA>
__global__ void k_scalars_to_ring(const double* __restrict__ reward, const uint8_t* __restrict__ done, int64_t n, int last_step_all,
                                  float* __restrict__ f_reward, float* __restrict__ f_done, float* __restrict__ f_last,
                                  float* __restrict__ f_avail, int64_t row0, int64_t cap) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        int64_t o = row0 + e; o = o >= cap ? o - cap : o;
        const float r = (float)reward[e];
        const float d = done[e] ? 1.0f : 0.0f;
        if (f_reward) {
#pragma unroll
            for (int a = 0; a < NA; ++a) f_reward[o * NA + a] = r;
        }
        if (f_done) f_done[o] = d;
        if (f_last) f_last[o] = (done[e] || last_step_all) ? 1.0f : 0.0f;      // done_ = done or t == max_steps - 1 (model.py:229)
        if (f_avail) {
#pragma unroll
            for (int j = 0; j < NA * POL_ACT; ++j) f_avail[o * (NA * POL_ACT) + j] = 1.0f;
        }
    }
}

// The small Transition fields of n envs in ONE launch (model.py:221, :229-242): action / log_prob_a rows, reward repeated per
// agent, done, last_step (= done, or every env when last_step_all), all-ones action_avail, and -- zero_values -- value /
// next_value as zeros (MADDPG's losses recompute both).  Thread = (env, column of the NA x 4 wide rows): coalesced throughout.
template <int NA>
__global__ void k_transition_tail(const float* __restrict__ action, const float* __restrict__ logp, const double* __restrict__ reward,
                                  const uint8_t* __restrict__ done, int64_t n, int last_step_all, int zero_values,
                                  float* __restrict__ f_action, float* __restrict__ f_logp, float* __restrict__ f_value,
                                  float* __restrict__ f_next_value, float* __restrict__ f_reward, float* __restrict__ f_done,
                                  float* __restrict__ f_last, float* __restrict__ f_avail, int64_t row0, int64_t cap) {
    constexpr int W = NA * POL_ACT;
    const int64_t total = n * W;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t e = i / W;
        const int c = (int)(i - e * W);
        int64_t o = row0 + e; o = o >= cap ? o - cap : o;
        f_action[o * W + c] = action[i];
        if (f_logp) f_logp[o * W + c] = logp[i];
        if (f_avail) f_avail[o * W + c] = 1.0f;
        if (c < NA) {
            f_reward[o * NA + c] = (float)reward[e];
            if (zero_values) { f_value[o * NA + c] = 0.0f; f_next_value[o * NA + c] = 0.0f; }
        }
        if (c == NA) { const bool d = done[e] != 0; f_done[o] = d ? 1.0f : 0.0f; f_last[o] = (d || last_step_all) ? 1.0f : 0.0f; }
    }
}

// MADDPG critic input (madrl/models/maddpg.py:29-66, shared parameters, agent_id): for batch row b and agent i
//   [ obs of all agents (NA x 144) | one-hot(i) (NA) | actions of all agents (NA x 4) ]   = 149 NA floats (745 for five agents)
template <int NA>
__global__ void k_critic_input(const float* __restrict__ state, const float* __restrict__ action, int64_t batch, float* __restrict__ out) {
    constexpr int W = NA * POL_OBS + NA + NA * POL_ACT;
    const int64_t total = batch * NA * W;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % W);
        const int64_t bi = i / W;
        const int ag = (int)(bi % NA);
        const int64_t b = bi / NA;
        float v;
        if (c < NA * POL_OBS) v = state[b * (NA * POL_OBS) + c];
        else if (c < NA * POL_OBS + NA) v = (c - NA * POL_OBS == ag) ? 1.0f : 0.0f;
        else v = action[b * (NA * POL_ACT) + (c - NA * POL_OBS - NA)];
        out[i] = v;
    }
}

// reward_normalisation (model.py:321-322): nn.BatchNorm1d(n_agents) in training mode with its initial affine
// parameters (weight 1, bias 0: the module is in no optimiser): per agent column, (x - mean) / sqrt(var_biased + 1e-5)
template <int NA>
__global__ void k_reward_batchnorm(const float* __restrict__ reward, int64_t batch, float* __restrict__ out) {
    const int a = blockIdx.x;                                       // one block per agent column
    __shared__ double sh[2][256];
    double s = 0.0, ss = 0.0;
    for (int64_t b = threadIdx.x; b < batch; b += blockDim.x) { const double x = reward[b * NA + a]; s += x; }
    sh[0][threadIdx.x] = s; __syncthreads();
    for (int d = 128; d > 0; d >>= 1) { if ((int)threadIdx.x < d) sh[0][threadIdx.x] += sh[0][threadIdx.x + d]; __syncthreads(); }
    const double mean = sh[0][0] / (double)batch;
    for (int64_t b = threadIdx.x; b < batch; b += blockDim.x) { const double x = reward[b * NA + a] - mean; ss += x * x; }
    sh[1][threadIdx.x] = ss; __syncthreads();
    for (int d = 128; d > 0; d >>= 1) { if ((int)threadIdx.x < d) sh[1][threadIdx.x] += sh[1][threadIdx.x + d]; __syncthreads(); }
    const double var = sh[1][0] / (double)batch;
    const float rstd = (float)(1.0 / sqrt(var + 1e-5)), meanf = (float)mean;
    for (int64_t b = threadIdx.x; b < batch; b += blockDim.x) out[b * NA + a] = (reward[b * NA + a] - meanf) * rstd;
}

int gt_grid(int64_t tiles, int per_sm) {       // persistent grid of the transposing gathers: per_sm CTAs per SM
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int64_t g = (int64_t)sms * per_sm;
    return (int)(tiles < g ? (tiles < 1 ? 1 : tiles) : g);
}

// One instantiation per agent count, indexed by the handle's na (entry 0 unused)
#define NA_TABLE(k) {nullptr, k<1>, k<2>, k<3>, k<4>, k<5>}
decltype(&k_policy<5>) const K_POLICY[POL_NA_MAX + 1] = NA_TABLE(k_policy);
decltype(&k_critic<5>) const K_CRITIC[POL_NA_MAX + 1] = NA_TABLE(k_critic);
decltype(&k_window_gather<5>) const K_WINDOW_GATHER[POL_NA_MAX + 1] = NA_TABLE(k_window_gather);
decltype(&k_em_gather<5>) const K_EM_GATHER[POL_NA_MAX + 1] = NA_TABLE(k_em_gather);
decltype(&k_scalars_to_ring<5>) const K_SCALARS_TO_RING[POL_NA_MAX + 1] = NA_TABLE(k_scalars_to_ring);
decltype(&k_transition_tail<5>) const K_TRANSITION_TAIL[POL_NA_MAX + 1] = NA_TABLE(k_transition_tail);
decltype(&k_critic_input<5>) const K_CRITIC_INPUT[POL_NA_MAX + 1] = NA_TABLE(k_critic_input);
decltype(&k_reward_batchnorm<5>) const K_REWARD_BATCHNORM[POL_NA_MAX + 1] = NA_TABLE(k_reward_batchnorm);
#undef NA_TABLE

float round_tf32(float x) {                    // round to nearest even on the 13 dropped mantissa bits
    uint32_t u; std::memcpy(&u, &x, 4);
    if ((u & 0x7F800000u) == 0x7F800000u) return x;
    u += 0x00000FFFu + ((u >> 13) & 1u);
    u &= 0xFFFFE000u;
    float y; std::memcpy(&y, &u, 4);
    return y;
}

}  // namespace

struct FpPolicy {
    int device = 0;
    int na = POL_NA_MAX;                           // agents per env, fixed at fp_policy_create_agents
    int loaded = 0;
    int attr_window = 0, attr_hidden = 0;          // opt-in shared-memory sizes of the gather kernels set on this handle's device
    float* d_W1rot = nullptr; float* d_Wg = nullptr; float* d_vec = nullptr;
    float* sink_out = nullptr; int64_t sink_pitch = 0, sink_row0 = 0, sink_cap = 0, sink_n = 0;   // fp_policy_state_sink: consumed by the next fp_policy_act
    int critic_loaded = 0;
    float* d_Wc1rot = nullptr; float* d_Wc2 = nullptr; float* d_Wca = nullptr; float* d_cvec = nullptr;   // critic (fp_critic_load)
    int64_t launches = 0;
    std::string err;
};

namespace {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {                  // the driver entry point, without linking libcuda
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}
}  // namespace

// The ring as a 3-D tensor [24 slots][na x 6 = agent x feature][n_pad envs] (innermost first); a tile is the box [24][6][128]
// at (env block, agent * 6, 0); envs past n_pad read as zeros.  Rings narrower than a tile: *use_tma = 0 (LDGSTS path).
static int ring_tensor_map(FpPolicy* p, const float* d_ring, int64_t n_pad, CUtensorMap* tmap, int32_t* use_tma, const char* who,
                           int box_slots = POL_H) {
    std::memset(tmap, 0, sizeof(*tmap));
    *use_tma = 0;
    if (n_pad >= POL_M && ((uintptr_t)d_ring & 15) == 0) {
        EncodeTiledFn enc = encode_tiled_fn();
        if (!enc) return fail(p, FP_ECUDA, std::string(who) + ": cuTensorMapEncodeTiled is not available from this driver");
        const cuuint64_t gdim[3] = {(cuuint64_t)n_pad, (cuuint64_t)(p->na * POL_F), (cuuint64_t)POL_H};
        const cuuint64_t gstride[2] = {(cuuint64_t)n_pad * 4, (cuuint64_t)n_pad * 4 * (p->na * POL_F)};
        const cuuint32_t box[3] = {POL_M, POL_F, (cuuint32_t)box_slots}, estr[3] = {1, 1, 1};
        const CUresult r = enc(tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(d_ring), gdim, gstride, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(p, FP_ECUDA, std::string(who) + ": cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
        *use_tma = 1;
    }
    return FP_OK;
}

extern "C" {

int fp_policy_create_agents(int device, int32_t n_agents, FpPolicy** out) {
    if (!out) return FP_EINVAL;
    if (n_agents < 1 || n_agents > POL_NA_MAX)
        return fail<FpPolicy>(nullptr, FP_EINVAL, "fp_policy_create_agents: n_agents must be in [1, 5], got " + std::to_string(n_agents));
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return fail<FpPolicy>(nullptr, FP_ECUDA, "fp_policy_create: no CUDA device (there is no CPU fallback)");
    if (device < 0 || device >= ndev) return fail<FpPolicy>(nullptr, FP_EINVAL, "fp_policy_create: bad device index");
    FpPolicy* p = new FpPolicy();
    p->device = device;
    p->na = n_agents;
    *out = p;
    return FP_OK;
}

int fp_policy_create(int device, FpPolicy** out) { return fp_policy_create_agents(device, POL_NA_MAX, out); }

int fp_policy_destroy(FpPolicy* p) {
    if (!p) return FP_OK;
    const DeviceGuard on_device(p->device);       // best effort: the handle is freed whatever happens
    cudaFree(p->d_W1rot); cudaFree(p->d_Wg); cudaFree(p->d_vec);
    cudaFree(p->d_Wc1rot); cudaFree(p->d_Wc2); cudaFree(p->d_Wca); cudaFree(p->d_cvec);
    delete p;
    return FP_OK;
}

const char* fp_policy_last_error(const FpPolicy* p) { return p ? p->err.c_str() : create_error<FpPolicy>().c_str(); }
int64_t fp_policy_launch_count(const FpPolicy* p) { return p ? p->launches : 0; }

// Host weights in torch's layouts (state_dict of RNNAgent, madrl/agents/rnn_agent.py:11-16):
//   fc1.weight [64][144 + na] (144 observation columns + na agent-id columns), fc1.bias [64], layernorm.weight / .bias [64],
//   rnn.weight_ih / weight_hh [192][64] (rows r | z | n), rnn.bias_ih / bias_hh [192], fc2.weight [4][64], fc2.bias [4]
int fp_policy_load(FpPolicy* p, const float* fc1_w, const float* fc1_b, const float* ln_g, const float* ln_b, const float* w_ih,
                   const float* w_hh, const float* b_ih, const float* b_hh, const float* fc2_w, const float* fc2_b) {
    if (!p) return FP_EINVAL;
    if (!fc1_w || !fc1_b || !ln_g || !ln_b || !w_ih || !w_hh || !b_ih || !b_hh || !fc2_w || !fc2_b)
        return fail(p, FP_EINVAL, "fp_policy_load: null weight array");
    USE_DEVICE(p);
    const int na = p->na, KIN = POL_OBS + na;
    // fc1: 24 column rotations, UMMA K-major layout [kc][n][4]; ring slot s holds history entry r = (s - q - 1) mod 24
    // when the newest slot is q, i.e. K index s * 6 + f must carry weight column r * 6 + f
    std::vector<float> W1((size_t)POL_H * POL_OBS * POL_HID, 0.0f);
    for (int q = 0; q < POL_H; ++q)
        for (int s = 0; s < POL_H; ++s) {
            const int r = ((s - q - 1) % POL_H + POL_H) % POL_H;
            for (int f = 0; f < POL_F; ++f) {
                const int k = s * POL_F + f, src = r * POL_F + f;
                for (int n = 0; n < POL_HID; ++n)
                    W1[(size_t)q * POL_OBS * POL_HID + ((size_t)(k >> 2) * POL_HID + n) * 4 + (k & 3)] = round_tf32(fc1_w[(size_t)n * KIN + src]);
            }
        }
    std::vector<float> Wg(WG_BYTES / 4, 0.0f), vec(V_FLOATS, 0.0f);
    {
        // gate rows permuted so that a column half holds, per quarter q (= worker thread of the row), the 8 units of chunk h with
        // their r and z outputs adjacent: rz packed row 64 h + 16 q + 8 g + j = gate row 64 g + 16 q + 8 h + j; n packed row
        // 32 h + 8 q + j = n-gate row 16 q + 8 h + j
        auto pack_rz = [](std::vector<float>& dst, size_t off, const float* w) {
            for (int np = 0; np < 128; ++np) {
                const int h = np >> 6, q = (np >> 4) & 3, g = (np >> 3) & 1, j = np & 7, n = 64 * g + 16 * q + 8 * h + j;
                for (int k = 0; k < POL_HID; ++k)
                    dst[off + ((size_t)(k >> 2) * 128 + np) * 4 + (k & 3)] = round_tf32(w[(size_t)n * POL_HID + k]);
            }
        };
        auto pack_n = [](std::vector<float>& dst, size_t off, const float* w) {
            for (int np = 0; np < 64; ++np) {
                const int h = np >> 5, q = (np >> 3) & 3, j = np & 7, n = 128 + 16 * q + 8 * h + j;
                for (int k = 0; k < POL_HID; ++k)
                    dst[off + ((size_t)(k >> 2) * 64 + np) * 4 + (k & 3)] = round_tf32(w[(size_t)n * POL_HID + k]);
            }
        };
        pack_rz(Wg, 0, w_ih);
        pack_rz(Wg, WG_RZ_BYTES / 4, w_hh);
        pack_n(Wg, 2 * WG_RZ_BYTES / 4, w_ih);
        pack_n(Wg, 2 * WG_RZ_BYTES / 4 + WG_N_BYTES / 4, w_hh);
    }
    for (int o = 0; o < POL_ACT; ++o)
        for (int k = 0; k < POL_HID; ++k) vec[V_W2 + 4 * k + o] = fc2_w[(size_t)o * POL_HID + k];      // fc2 runs in fp32: unrounded
    for (int a = 0; a < na; ++a)
        for (int n = 0; n < POL_HID; ++n) vec[V_B1A + a * POL_HID + n] = fc1_b[n] + fc1_w[(size_t)n * KIN + POL_OBS + a];   // one-hot column folded in
    for (int n = 0; n < POL_HID; ++n) { vec[V_LNG + n] = ln_g[n]; vec[V_LNB + n] = ln_b[n]; }
    // gate biases in the exponential's unit (see sigmoid8 / tanh8_scaled)
    for (int n = 0; n < POL_HID; ++n) {
        vec[V_BIN + n] = (float)((double)b_ih[128 + n] * (2.0 * (double)POL_L2E)); vec[V_BHN + n] = (float)((double)b_hh[128 + n] * (2.0 * (double)POL_L2E));
    }
    for (int n = 0; n < 128; ++n) vec[V_BRZ + n] = (float)(-((double)b_ih[n] + (double)b_hh[n]) * (double)POL_L2E);
    for (int n = 0; n < POL_ACT; ++n) vec[V_B2 + n] = fc2_b[n];
    p->loaded = 0;
    cudaFree(p->d_W1rot); cudaFree(p->d_Wg); cudaFree(p->d_vec);
    p->d_W1rot = p->d_Wg = p->d_vec = nullptr;
    CUDA_TRY(p, alloc_group({{&p->d_W1rot, W1.size() * 4}, {&p->d_Wg, Wg.size() * 4}, {&p->d_vec, vec.size() * 4}}));
    CUDA_TRY(p, cudaMemcpy(p->d_W1rot, W1.data(), W1.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(p, cudaMemcpy(p->d_Wg, Wg.data(), Wg.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(p, cudaMemcpy(p->d_vec, vec.data(), vec.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(p, cudaFuncSetAttribute(K_POLICY[na], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)POL_SMEM));
    p->loaded = 1;
    return FP_OK;
}

// One acting step for n_envs x na agents (na = the handle's agent count).  d_ring / slot / n_pad: the observation ring (fp_obs_ring, fp_step_ring).
// d_hid_in (may be null = zeros) / d_hid_out: [n_envs][na][64] (or env-minor [na][64][n_pad]); d_reset (may be null): envs whose hidden state restarts
// at zero (init_hidden, model.py:211).  d_mean, d_logp may be null.  explore = 1: status 'train' with exploration
// (d_eps = caller-supplied standard-normal draws [n_envs][na][4], or null: Philox keyed by (seed, row, step));
// explore = 0: status 'test'.  std = fixed_policy_std (default.yaml: 1.0).
int fp_policy_act(FpPolicy* p, const float* d_ring, int32_t slot, int64_t n_pad, int64_t n_envs, const float* d_hid_in,
                  const uint8_t* d_reset, float* d_hid_out, int32_t hid_env_minor, float* d_mean, float* d_action, float* d_logp,
                  const float* d_eps, uint64_t seed, uint64_t step, float std_, int32_t explore, void* stream) {
    if (!p) return FP_EINVAL;
    if (!p->loaded) return fail(p, FP_ESTATE, "fp_policy_act: call fp_policy_load first");
    if (!d_ring || !d_hid_out || !d_action || n_envs < 1 || slot < 0 || slot >= POL_H || n_pad < n_envs || (n_pad & 3))
        return fail(p, FP_EINVAL, "fp_policy_act: bad arguments");
    if (!(std_ > 0.0f)) return fail(p, FP_EINVAL, "fp_policy_act: std must be positive");
    USE_DEVICE(p);
    PolParams prm;
    std::memset(&prm, 0, sizeof(prm));
    prm.ring = d_ring; prm.n_pad = n_pad; prm.n = n_envs; prm.slot = slot;
    prm.W1rot = p->d_W1rot; prm.Wg = p->d_Wg; prm.vec = p->d_vec;
    prm.hid_in = d_hid_in; prm.reset = d_reset; prm.hid_out = d_hid_out; prm.hid_em = hid_env_minor ? 1 : 0;
    prm.mean = d_mean; prm.action = d_action; prm.logp = d_logp; prm.eps = d_eps;
    prm.seed = seed; prm.step = step; prm.std_ = std_; prm.log_std = std::log(std_); prm.explore = explore;
    alignas(64) CUtensorMap tmap;
    { const int rc = ring_tensor_map(p, d_ring, n_pad, &tmap, &prm.use_tma, "fp_policy_act"); if (rc != FP_OK) return rc; }
    if (p->sink_out) {                                  // one-shot `state` sink (fp_policy_state_sink); needs the TMA path
        if (!prm.use_tma || p->sink_n > n_envs) { p->sink_out = nullptr; return fail(p, FP_EINVAL, "fp_policy_act: the state sink needs n_pad >= 128 and at most n_envs rows"); }
        prm.st_out = p->sink_out; prm.st_pitch = p->sink_pitch; prm.st_row0 = p->sink_row0; prm.st_cap = p->sink_cap; prm.st_n = p->sink_n;
        p->sink_out = nullptr;
    }
    int sms = 0;
    CUDA_TRY(p, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, p->device));
    const int64_t tiles = (n_envs + POL_M - 1) / POL_M * p->na;
    const int grid = (int)(tiles < sms ? tiles : sms);
    K_POLICY[p->na]<<<grid, POL_THREADS, POL_SMEM, (cudaStream_t)stream>>>(prm, tmap);
    return launched(p, "k_policy");
}

// select_action alone on stored fc2 outputs d_mean [n_envs][na][4] (fp_policy_act's d_mean): another exploration draw of the
// same policy evaluation (same arguments as fp_policy_act's sampling part; bit-identical to re-running it with these draws).
int fp_policy_sample(FpPolicy* p, const float* d_mean, int64_t n_envs, float* d_action, float* d_logp, const float* d_eps,
                     uint64_t seed, uint64_t step, float std_, int32_t explore, void* stream) {
    if (!p) return FP_EINVAL;
    if (!d_mean || !d_action || n_envs < 1) return fail(p, FP_EINVAL, "fp_policy_sample: bad arguments");
    if (!(std_ > 0.0f)) return fail(p, FP_EINVAL, "fp_policy_sample: std must be positive");
    USE_DEVICE(p);
    k_sample<<<grid_for(n_envs * p->na), 256, 0, (cudaStream_t)stream>>>(d_mean, n_envs * p->na, explore, d_eps, seed, step, std_, std::log(std_),
                                                                          d_action, d_logp);
    return launched(p, "k_sample");
}

// One-shot sink for the NEXT fp_policy_act: while it evaluates the policy, its writer warps copy the dense get_obs windows
// [na][144] of envs [0, n) -- the very blocks the kernel has staged -- into rows (row0 + e) mod cap of pitch `pitch` floats: the
// Transition's `state` (model.py:230-237) without a separate pass over the ring (fp_policy_gather_windows).  Needs a ring of
// at least 128 envs (n_pad >= 128).
int fp_policy_state_sink(FpPolicy* p, float* d_field, int64_t pitch, int64_t row0, int64_t cap, int64_t n) {
    if (!p) return FP_EINVAL;
    if (!d_field || n < 1 || pitch < p->na * POL_OBS || (pitch & 3) || ((uintptr_t)d_field & 15) || row0 < 0 || cap < n || row0 >= cap)
        return fail(p, FP_EINVAL, "fp_policy_state_sink: bad arguments");
    p->sink_out = d_field; p->sink_pitch = pitch; p->sink_row0 = row0; p->sink_cap = cap; p->sink_n = n;
    return FP_OK;
}

// Dense observation windows of envs [0, n) (get_obs layout [n][na][144], oldest entry first) from the ring into rows
// (row0 + e) mod cap of pitch `pitch` floats: a replay field (state / next_state of the Transition, model.py:230-237)
// or, with row0 = 0 and cap >= n, a dense tensor.
int fp_policy_gather_windows(FpPolicy* p, const float* d_ring, int32_t slot, int64_t n_pad, int64_t n, float* d_out, int64_t pitch,
                             int64_t row0, int64_t cap, void* stream) {
    if (!p) return FP_EINVAL;
    if (!d_ring || !d_out || n < 1 || pitch < p->na * POL_OBS || row0 < 0 || cap < n || row0 >= cap || slot < 0 || slot >= POL_H)
        return fail(p, FP_EINVAL, "fp_policy_gather_windows: bad arguments");
    USE_DEVICE(p);
    constexpr int smem_w = POL_OBS * GT_STRIDE * (int)sizeof(float);
    if (!p->attr_window) { CUDA_TRY(p, cudaFuncSetAttribute(K_WINDOW_GATHER[p->na], cudaFuncAttributeMaxDynamicSharedMemorySize, smem_w)); p->attr_window = 1; }
    K_WINDOW_GATHER[p->na]<<<gt_grid(((n + GT_ENVS - 1) / GT_ENVS) * p->na, 3), 256, smem_w, (cudaStream_t)stream>>>(d_ring, n_pad, slot, n, d_out, pitch, row0, cap);
    return launched(p, "k_window_gather");
}

// Hidden states in the policy kernel's env-minor layout [na][64][n_pad] -> replay rows (last_hid / hid, na x 64 floats per env);
// d_zero_mask (may be null): envs whose row is written as zeros (a restarted env's last_hid is the zero state it acted from)
int fp_policy_hidden_to_ring(FpPolicy* p, const float* d_hid_em, int64_t n_pad, int64_t n, float* d_field, int64_t row0, int64_t cap,
                             const uint8_t* d_zero_mask, void* stream) {
    if (!p) return FP_EINVAL;
    if (!d_hid_em || !d_field || n < 1 || n_pad < n || row0 < 0 || cap < n || row0 >= cap) return fail(p, FP_EINVAL, "fp_policy_hidden_to_ring: bad arguments");
    USE_DEVICE(p);
    const int smem_h = p->na * POL_HID / 2 * GT_STRIDE * (int)sizeof(float);        // [na x 64 / 2][129]
    if (!p->attr_hidden) { CUDA_TRY(p, cudaFuncSetAttribute(K_EM_GATHER[p->na], cudaFuncAttributeMaxDynamicSharedMemorySize, smem_h)); p->attr_hidden = 1; }
    K_EM_GATHER[p->na]<<<gt_grid(((n + GT_ENVS - 1) / GT_ENVS) * 2, 2), 256, smem_h, (cudaStream_t)stream>>>(d_hid_em, n_pad, n, d_field, row0, cap, d_zero_mask);
    return launched(p, "k_em_gather");
}

int fp_policy_rows_to_ring(FpPolicy* p, const float* d_src, int64_t n, int32_t width, float* d_field, int64_t row0, int64_t cap, void* stream) {
    if (!p) return FP_EINVAL;
    if (!d_src || !d_field || n < 1 || width < 1 || row0 < 0 || cap < n || row0 >= cap) return fail(p, FP_EINVAL, "fp_policy_rows_to_ring: bad arguments");
    USE_DEVICE(p);
    k_rows_to_ring<<<grid_for(n * width), 256, 0, (cudaStream_t)stream>>>(d_src, n, width, d_field, row0, cap);
    return launched(p, "k_rows_to_ring");
}

int fp_policy_scalars_to_ring(FpPolicy* p, const double* d_reward, const uint8_t* d_done, int64_t n, int32_t last_step_all,
                              float* f_reward, float* f_done, float* f_last, float* f_avail, int64_t row0, int64_t cap, void* stream) {
    if (!p) return FP_EINVAL;
    if (!d_reward || !d_done || n < 1 || row0 < 0 || cap < n || row0 >= cap) return fail(p, FP_EINVAL, "fp_policy_scalars_to_ring: bad arguments");
    USE_DEVICE(p);
    K_SCALARS_TO_RING[p->na]<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(d_reward, d_done, n, last_step_all, f_reward, f_done, f_last, f_avail, row0, cap);
    return launched(p, "k_scalars_to_ring");
}

int fp_policy_transition_tail(FpPolicy* p, const float* d_action, const float* d_logp, const double* d_reward, const uint8_t* d_done,
                              int64_t n, int32_t last_step_all, int32_t zero_values, float* f_action, float* f_logp, float* f_value,
                              float* f_next_value, float* f_reward, float* f_done, float* f_last, float* f_avail, int64_t row0,
                              int64_t cap, void* stream) {
    if (!p) return FP_EINVAL;
    if (!d_action || !d_reward || !d_done || !f_action || !f_reward || !f_done || !f_last || (f_logp && !d_logp) ||
        (zero_values && (!f_value || !f_next_value)) || n < 1 || row0 < 0 || cap < n || row0 >= cap)
        return fail(p, FP_EINVAL, "fp_policy_transition_tail: bad arguments");
    USE_DEVICE(p);
    K_TRANSITION_TAIL[p->na]<<<grid_for(n * p->na * POL_ACT), 256, 0, (cudaStream_t)stream>>>(d_action, d_logp, d_reward, d_done, n, last_step_all,
                                                                                       zero_values, f_action, f_logp, f_value, f_next_value,
                                                                                       f_reward, f_done, f_last, f_avail, row0, cap);
    return launched(p, "k_transition_tail");
}

// Critic weights, HOST fp32 arrays in torch's state_dict layouts (MLPCritic, madrl/critics/mlp_critic.py:5-20, as
// MADDPG.construct_value_net builds it, maddpg.py:18-27): fc1.weight [64][149 na] (144 na observation columns | na agent-id
// columns | 4 na action columns), fc1.bias [64], layernorm.weight / .bias [64], fc2.weight [64][64], fc2.bias [64], fc3.weight [1][64],
// fc3.bias [1].
int fp_critic_load(FpPolicy* p, const float* fc1_w, const float* fc1_b, const float* ln_g, const float* ln_b, const float* fc2_w,
                   const float* fc2_b, const float* fc3_w, const float* fc3_b) {
    if (!p) return FP_EINVAL;
    if (!fc1_w || !fc1_b || !ln_g || !ln_b || !fc2_w || !fc2_b || !fc3_w || !fc3_b) return fail(p, FP_EINVAL, "fp_critic_load: null weight array");
    USE_DEVICE(p);
    const int na = p->na, KIN = na * POL_OBS + na + na * POL_ACT;          // 149 na: 745 for five agents
    const size_t blk = CR_WB_BYTES / 4;
    // fc1, observation columns: per ring rotation q and agent block a, UMMA K-major layout [kc][n][4] (see fp_policy_load)
    std::vector<float> W1((size_t)POL_H * na * blk, 0.0f);
    for (int q = 0; q < POL_H; ++q)
        for (int a = 0; a < na; ++a)
            for (int sl = 0; sl < POL_H; ++sl) {
                const int r = ((sl - q - 1) % POL_H + POL_H) % POL_H;
                for (int f = 0; f < POL_F; ++f) {
                    const int k = sl * POL_F + f, src = a * POL_OBS + r * POL_F + f;
                    for (int n = 0; n < POL_HID; ++n)
                        W1[((size_t)q * na + a) * blk + ((size_t)(k >> 2) * POL_HID + n) * 4 + (k & 3)] = round_tf32(fc1_w[(size_t)n * KIN + src]);
                }
            }
    std::vector<float> W2(CR_W2_BYTES / 4, 0.0f), Wa(CR_WA_BYTES / 4, 0.0f), vec(CV_FLOATS, 0.0f);
    for (int n = 0; n < POL_HID; ++n) {
        for (int k = 0; k < POL_HID; ++k) W2[((size_t)(k >> 2) * POL_HID + n) * 4 + (k & 3)] = round_tf32(fc2_w[(size_t)n * POL_HID + k]);
        for (int k = 0; k < na * POL_ACT; ++k)
            Wa[((size_t)(k >> 2) * POL_HID + n) * 4 + (k & 3)] = round_tf32(fc1_w[(size_t)n * KIN + na * POL_OBS + na + k]);
        for (int a = 0; a < na; ++a) vec[CV_B1A + a * POL_HID + n] = fc1_b[n] + fc1_w[(size_t)n * KIN + na * POL_OBS + a];   // one-hot column folded in
        vec[CV_LNG + n] = ln_g[n]; vec[CV_LNB + n] = ln_b[n]; vec[CV_B2 + n] = fc2_b[n]; vec[CV_W3 + n] = fc3_w[n];           // fc3 runs in fp32: unrounded
    }
    vec[CV_B3] = fc3_b[0];
    p->critic_loaded = 0;
    cudaFree(p->d_Wc1rot); cudaFree(p->d_Wc2); cudaFree(p->d_Wca); cudaFree(p->d_cvec);
    p->d_Wc1rot = p->d_Wc2 = p->d_Wca = p->d_cvec = nullptr;
    CUDA_TRY(p, alloc_group({{&p->d_Wc1rot, W1.size() * 4}, {&p->d_Wc2, W2.size() * 4}, {&p->d_Wca, Wa.size() * 4},
                             {&p->d_cvec, vec.size() * 4}}));
    CUDA_TRY(p, cudaMemcpy(p->d_Wc1rot, W1.data(), W1.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(p, cudaMemcpy(p->d_Wc2, W2.data(), W2.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(p, cudaMemcpy(p->d_Wca, Wa.data(), Wa.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(p, cudaMemcpy(p->d_cvec, vec.data(), vec.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(p, cudaFuncSetAttribute(K_CRITIC[na], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CR_SMEM));
    p->critic_loaded = 1;
    return FP_OK;
}

// MADDPG.value (maddpg.py:29-76) for n_envs envs: d_value[n_envs][na] = the critic on (the observation ring's windows of all
// agents, agent id, d_actions[n_envs][na][4]) -- the Transition's value (model.py:217) or, on the ring after the step and a
// second sampled action, next_value (:225-226).
int fp_critic_value(FpPolicy* p, const float* d_ring, int32_t slot, int64_t n_pad, int64_t n_envs, const float* d_actions,
                    float* d_value, void* stream) {
    if (!p) return FP_EINVAL;
    if (!p->critic_loaded) return fail(p, FP_ESTATE, "fp_critic_value: call fp_critic_load first");
    if (!d_ring || !d_actions || !d_value || n_envs < 1 || slot < 0 || slot >= POL_H || n_pad < n_envs || (n_pad & 3))
        return fail(p, FP_EINVAL, "fp_critic_value: bad arguments");
    USE_DEVICE(p);
    CritParams prm;
    std::memset(&prm, 0, sizeof(prm));
    prm.ring = d_ring; prm.n_pad = n_pad; prm.n = n_envs; prm.slot = slot;
    prm.Wc1rot = p->d_Wc1rot; prm.W2 = p->d_Wc2; prm.Wa = p->d_Wca; prm.vec = p->d_cvec;
    prm.actions = d_actions; prm.value = d_value;
    alignas(64) CUtensorMap tmap;
    { const int rc = ring_tensor_map(p, d_ring, n_pad, &tmap, &prm.use_tma, "fp_critic_value", POL_H / 2); if (rc != FP_OK) return rc; }   // half-block boxes
    int sms = 0;
    CUDA_TRY(p, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, p->device));
    const int64_t tiles = (n_envs + POL_M - 1) / POL_M;
    const int grid = (int)(tiles < sms ? tiles : sms);
    K_CRITIC[p->na]<<<grid, CRIT_THREADS, CR_SMEM, (cudaStream_t)stream>>>(prm, tmap);
    return launched(p, "k_critic");
}

// Learner feed (unpack_data, madrl/models/model.py:308-323, on a sampled batch already on the device):
//   d_critic_in [batch * na][149 na]: the MADDPG critic's input rows (maddpg.py:29-66); d_reward_norm [batch][na]: the
//   reward after reward_normalisation (BatchNorm1d over the batch, training mode).  Either may be null.
int fp_learner_feed(FpPolicy* p, const float* d_state, const float* d_action, const float* d_reward, int64_t batch,
                    float* d_critic_in, float* d_reward_norm, void* stream) {
    if (!p) return FP_EINVAL;
    if (batch < 1 || (d_critic_in && (!d_state || !d_action)) || (d_reward_norm && !d_reward)) return fail(p, FP_EINVAL, "fp_learner_feed: bad arguments");
    USE_DEVICE(p);
    if (d_critic_in)
        K_CRITIC_INPUT[p->na]<<<grid_for(batch * p->na * (p->na * (POL_OBS + 1 + POL_ACT))), 256, 0, (cudaStream_t)stream>>>(d_state, d_action, batch, d_critic_in);
    if (d_reward_norm) K_REWARD_BATCHNORM[p->na]<<<p->na, 256, 0, (cudaStream_t)stream>>>(d_reward, batch, d_reward_norm);
    return launched(p, "fp_learner_feed", (d_critic_in != nullptr) + (d_reward_norm != nullptr));
}

}  // extern "C"
