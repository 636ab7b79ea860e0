// flex_common.cuh -- device-side structures and the warp-per-env DistFlow sweep.
//
// One warp owns one environment; lane k owns line k (the line feeding the bus whose DFS
// pre-order rank is k+1).  Pre-order numbering makes every subtree a contiguous lane range
// [k, end_k], so
//   * the backward sweep  (utils/pf.py:65-83: P_ij = p_j + sum_children(P_jk + R_jk l_jk))
//     is an inclusive warp scan followed by one indexed shuffle:  P_k = p_k + (S[end_k] - S[k]);
//   * the forward sweep   (utils/pf.py:90-94: v_j = v_i - 2(R P + X Q) - |z|^2 l)
//     is a root-path sum by pointer jumping over the statically known 2^r-th ancestors;
//   * the current update  (utils/pf.py:85-88: l v_j = P^2 + Q^2) is one IEEE fp64 divide/lane.
//
// All arithmetic is fp64 with a FIXED operation order (compiled with -fmad=false; fused
// multiply-adds are written explicitly as fma()) so that oracle/c/flex_oracle.c can mirror
// it bit for bit -- that is what makes the voltage-violation masks bit-exact.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/flexgpu.h"

#define FULL 0xffffffffu
#define FP_NL 32            // lanes == max lines
#define ANC_NONE 32u

// Scalar configuration, passed by value as a kernel parameter (uniform constant-bank reads).
struct DevCfg {
    int32_t nb, nl, na, history, episode_limit, raw_actions, pf_max_iter, obs_w;
    double pf_tol, v_min, v_max, e_min, e_max, p_ch_max, p_dis_max, eta_ch, eta_dis, inv_eta_dis, inv_eta_ch;
    double mpr, kappa, pv_cost, ess_cost, discomfort_coeff, voltage_coeff, delta_t, fail_penalty;
    double e_next_lb, slack_pen;
    int32_t slack_viol, pf_f32;      // pf_f32: opening passes of the thread kernels' solve that run in fp32
};

// Per-lane topology tables.  Lives in global memory (handle-owned); every CTA stages it into
// shared memory once and each lane then keeps its own hot entries (R, X, |z|^2, end, anc) in
// registers for the whole grid-stride loop.
struct DevTopo {
    double R[FP_NL], X[FP_NL], Z2[FP_NL], imax2[FP_NL];
    int32_t end[FP_NL];        // last lane of this lane's subtree
    uint32_t anc[FP_NL];       // 5 x 6-bit: lane of the 2^r-th ancestor line, ANC_NONE if none
    int32_t col[FP_NL];        // dataset column (= bus position - 1) of this lane's bus
    int32_t agent[FP_NL];      // agent whose building sits on this lane's bus, else -1
    int32_t agent_lane[8];     // lane of agent i's bus
    int32_t agent_col[8];      // dataset column of agent i's bus
};

// Topology tables of the thread-per-env kernels.  Passed BY VALUE inside the kernel parameter
// block: after full unrolling every entry is a compile-time offset into the constant bank, so
// impedances feed DFMA directly as constant operands and the flags become uniform predicates.
// "Slots" are per-thread shared-memory cells for the few buses with more than one child
// (IEEE-33: buses 2, 3, 6): the parent voltage for non-adjacent children (forward sweep) and
// the accumulated contributions of non-adjacent children (backward sweep).
#define FP_MAX_SLOTS 8
#define TT_ROOT (-1)         // par_src: the slack bus feeds this line (v_parent = 1)
#define TT_CARRY (-2)        // par_src / dep_slot: parent is lane k-1 -> value carried in a register
#define FP_MAX_CHAINS 16
struct ThreadTopo {
    double R[FP_NL], X[FP_NL], Z2h[FP_NL], imax2[FP_NL];      // Z2h = |z|^2 / 2 (exact scaling)
    float Rf[FP_NL], Xf[FP_NL], Z2hf[FP_NL];                   // the same, rounded to fp32 (opening passes)
    int8_t par_src[FP_NL];    // forward: TT_ROOT, TT_CARRY or the slot holding v_parent
    int8_t own_slot[FP_NL];   // slot owned by this lane's bus (it has non-adjacent children), else -1
    int8_t dep_slot[FP_NL];   // backward: TT_ROOT (nothing), TT_CARRY (to lane k-1) or slot to deposit into
    int8_t dep_first[FP_NL];  // first deposit into that slot in a backward pass (store, not add)
    int8_t next_is_child[FP_NL];  // parent(lane k+1) == lane k
    int8_t chain_of[FP_NL];   // chain (maximal first-child path) this lane belongs to; chain 0 starts at lane 0
    int8_t col[FP_NL];        // dataset column (bus position - 1) of this lane's bus
    int8_t lane_of_col[FP_NL];
    int8_t agent_lane[8], agent_col[8];
    uint16_t attach_mask[FP_NL];          // chains whose head line leaves this lane's bus (non-adjacent children)
    uint16_t child_mask[FP_MAX_CHAINS];   // chains attached to any lane of this chain
    int32_t nl, n_slots, any_imax, n_chains;
};

// Slot / carry tables derived from the DFS parent-lane array.  constexpr: evaluated at compile
// time for the built-in shapes and at run time (host) for any other radial feeder.
struct TreeTables {
    int8_t par_src[FP_NL], own_slot[FP_NL], dep_slot[FP_NL], dep_first[FP_NL], next_is_child[FP_NL], chain_of[FP_NL];
    uint16_t attach_mask[FP_NL], child_mask[FP_NL];
    int n_slots, n_chains;
};

template <class ParArray>
constexpr TreeTables derive_tree_tables(const ParArray& par, int nl) {
    TreeTables t{};
    for (int k = 0; k < FP_NL; ++k) {
        t.par_src[k] = TT_ROOT; t.own_slot[k] = -1; t.dep_slot[k] = TT_ROOT; t.dep_first[k] = 0; t.next_is_child[k] = 0;
        t.chain_of[k] = 0; t.attach_mask[k] = 0; t.child_mask[k] = 0;
    }
    t.n_slots = 0; t.n_chains = 0;
    // chains: a lane whose parent is not lane k-1 (a lateral's first line, or a line leaving the slack
    // bus) starts a new chain; pre-order numbering gives nested chains larger ids than their hosts
    for (int k = 0; k < nl; ++k) {
        if (k == 0 || par[k] != k - 1) {
            const int c = t.n_chains++;
            t.chain_of[k] = (int8_t)c;
            if (par[k] >= 0 && c < 16) {
                t.attach_mask[par[k]] = (uint16_t)(t.attach_mask[par[k]] | (1u << c));
                t.child_mask[t.chain_of[par[k]]] = (uint16_t)(t.child_mask[t.chain_of[par[k]]] | (1u << c));
            }
        } else {
            t.chain_of[k] = t.chain_of[k - 1];
        }
    }
    for (int a = 0; a < nl; ++a) {                       // slots in increasing lane order of their owner
        bool has = false;
        for (int j = a + 2; j < nl; ++j) if (par[j] == a) has = true;
        if (has) t.own_slot[a] = (int8_t)t.n_slots++;
    }
    for (int j = 0; j < nl; ++j) {
        const int a = par[j];
        if (a < 0) continue;
        if (a == j - 1) { t.par_src[j] = TT_CARRY; t.dep_slot[j] = TT_CARRY; t.next_is_child[a] = 1; }
        else {
            t.par_src[j] = t.own_slot[a]; t.dep_slot[j] = t.own_slot[a];
            bool later = false;                          // reverse pre-order: the highest lane deposits first
            for (int m = j + 1; m < nl; ++m) if (par[m] == a) later = true;
            t.dep_first[j] = later ? 0 : 1;
        }
    }
    return t;
}

// IEEE 33-bus feeder (Baran & Wu), DFS pre-order with children in ascending bus position:
// lanes 0-16 = buses 2..18, 17-24 = buses 26..33 (off bus 6), 25-27 = buses 23..25 (off bus 3),
// 28-31 = buses 19..22 (off bus 2).
struct Ieee33Tree {
    static constexpr int NL = 32;
    static constexpr int8_t PAR[FP_NL] = {-1, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15,
                                          4, 17, 18, 19, 20, 21, 22, 23, 1, 25, 26, 0, 28, 29, 30};
    static constexpr int8_t COL[FP_NL] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16,
                                          24, 25, 26, 27, 28, 29, 30, 31, 21, 22, 23, 17, 18, 19, 20};
    // emission order of the unrolled sweeps (parents before children): main feeder (chain 0)
    // interleaved with the three laterals (chain 1), each lateral after its branch bus
    static constexpr int8_t ORDER[FP_NL] = {0, 1, 28, 2, 29, 3, 30, 4, 31, 5, 25, 6, 26, 7, 27, 8, 17,
                                            9, 18, 10, 19, 11, 20, 12, 21, 13, 22, 14, 23, 15, 24, 16};
    static constexpr int8_t CHAIN[FP_NL] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,
                                            1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1};
};
enum { SHAPE_RUNTIME = 0, SHAPE_IEEE33 = 1 };

struct LaneTopo {
    double R, X, Z2;
    int32_t end;
    uint32_t anc;
};

__device__ __forceinline__ LaneTopo load_lane_topo(const DevTopo& t, int lane) {
    LaneTopo l;
    l.R = t.R[lane]; l.X = t.X[lane]; l.Z2 = t.Z2[lane];
    l.end = t.end[lane]; l.anc = t.anc[lane];
    return l;
}

__device__ __forceinline__ void stage_topo(DevTopo* s_topo, const DevTopo* __restrict__ g_topo) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(g_topo);
    uint32_t* dst = reinterpret_cast<uint32_t*>(s_topo);
    for (int i = threadIdx.x; i < (int)(sizeof(DevTopo) / 4); i += blockDim.x) dst[i] = src[i];
    __syncthreads();
}

// two int32 fields of one 64-bit record word: lo in the low half
__device__ __forceinline__ uint64_t pack2(int32_t lo, int32_t hi) {
    return (uint64_t)(uint32_t)lo | ((uint64_t)(uint32_t)hi << 32);
}

// numpy.clip for a non-NaN x (the same two selects, signed zeros included), but a NaN x returns lo where numpy keeps
// the NaN.  The step kernels test their actions for NaN themselves (a NaN action is a solver failure and rolls the env
// back), so what the clip makes of one never reaches their outputs; clip_np is the exact numpy.clip.
__device__ __forceinline__ double clipd(double x, double lo, double hi) {
    double t = (x > lo) ? x : lo;
    return (t < hi) ? t : hi;
}

// numpy.clip exactly (_NPY_CLIP: minimum(maximum(x, lo), hi), a NaN x propagates): the safety layer's parse_actions
__device__ __forceinline__ double clip_np(double x, double lo, double hi) {
    return (x != x) ? x : clipd(x, lo, hi);
}

// Inclusive Hillis-Steele scan over the warp (lane order).
__device__ __forceinline__ double warp_scan_incl(double s, int lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        double y = __shfl_up_sync(FULL, s, d);
        if (lane >= d) s = s + y;
    }
    return s;
}

// Butterfly sum; every lane ends with the same value.
__device__ __forceinline__ double warp_sum_xor(double s) {
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) s = s + __shfl_xor_sync(FULL, s, d);
    return s;
}

struct SweepOut {
    double P, Q, ell, v;   // receiving-end flows, squared current, squared voltage of this lane
    int iters;
    bool ok;
};

// Backward/forward sweep from a flat start (l = 0, v = 1).  p, q: net consumption at this
// lane's bus.  Lanes >= nl must pass p = q = 0 and a LaneTopo with R = X = Z2 = 0, end = lane,
// anc = none (the host builds the tables that way).
__device__ __forceinline__ SweepOut distflow_sweep(const LaneTopo& t, double p, double q, int lane,
                                                  double tol, int max_iter, bool inject_fail) {
    SweepOut o;
    double ell = 0.0, v_old = 1.0, P = 0.0, Q = 0.0, v = 1.0;
    bool conv = false, bad = false;
    int it = 0;
    while (it < max_iter) {
        ++it;
        // ---- backward: subtree sums of x = p + R*l (sending-end contributions)
        double SP = warp_scan_incl(fma(t.R, ell, p), lane);
        double SQ = warp_scan_incl(fma(t.X, ell, q), lane);
        double SPe = __shfl_sync(FULL, SP, t.end);
        double SQe = __shfl_sync(FULL, SQ, t.end);
        P = p + (SPe - SP);
        Q = q + (SQe - SQ);
        // ---- forward: v = 1 - sum over the root path of the per-line drops
        double d = t.R * P;
        d = fma(t.X, Q, d);
        d = fma(t.Z2, ell, d + d);
#pragma unroll
        for (int r = 0; r < 5; ++r) {
            uint32_t a = (t.anc >> (6 * r)) & 63u;
            double y = __shfl_sync(FULL, d, a & 31u);
            if (a < ANC_NONE) d = d + y;
        }
        v = 1.0 - d;
        // ---- current: l = (P^2 + Q^2) / v
        double s = P * P;
        s = fma(Q, Q, s);
        ell = s / v;
        bad = __any_sync(FULL, !(v > 0.0));
        conv = __all_sync(FULL, fabs(v - v_old) <= tol);
        v_old = v;
        if (bad || conv) break;
    }
    o.P = P; o.Q = Q; o.ell = ell; o.v = v; o.iters = it;
    o.ok = conv && !bad && !inject_fail;
    return o;
}

// ------------------------------------------------------------------ reciprocal seed (thread / pair kernels)
// fp64 <-> fp32 by integer bit manipulation instead of F2F: the conversions are quarter-rate,
// ~18-cycle, scoreboard-tracked instructions on the XU pipe, and a warp has six scoreboards for
// everything of variable latency -- two conversions per line were what kept lines from
// overlapping.  Valid for positive normal values inside the fp32 range (squared voltages are
// ~1); anything else is caught by sqv_bad() or fails to converge and is reported as a failed solve.
//   d2f_trunc  truncates (a seed does not care), f2d_exact is exact
__device__ __forceinline__ float d2f_trunc(double v) {
    return __int_as_float(__funnelshift_l((unsigned)__double2loint(v), (unsigned)(__double2hiint(v) - 0x38000000), 3));
}
__device__ __forceinline__ double f2d_exact(float x) {
    const unsigned b = __float_as_uint(x);
    return __hiloint2double((int)((b >> 3) + 0x38000000u), (int)(b << 29));
}
// v <= 0 (also -0 and the smallest denormals), +-inf or NaN: one unsigned compare on the high word
__device__ __forceinline__ bool sqv_bad(double v) { return (unsigned)(__double2hiint(v) - 1) >= 0x7FEFFFFFu; }

// ------------------------------------------------------------------ Philox4x32-10
struct U4 { uint32_t x, y, z, w; };

__host__ __device__ __forceinline__ U4 philox4x32_10(U4 c, uint32_t k0, uint32_t k1) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)M0 * c.x, p1 = (uint64_t)M1 * c.z;
        U4 n;
        n.x = (uint32_t)(p1 >> 32) ^ c.y ^ k0;
        n.y = (uint32_t)p1;
        n.z = (uint32_t)(p0 >> 32) ^ c.w ^ k1;
        n.w = (uint32_t)p0;
        c = n;
        k0 += W0; k1 += W1;
    }
    return c;
}

// 53-bit uniform in [0,1) from two 32-bit words (same construction as numpy's random_sample).
__host__ __device__ __forceinline__ double u53(uint32_t a, uint32_t b) {
    return (double)(((uint64_t)(a >> 5) << 26) | (uint64_t)(b >> 6)) * (1.0 / 9007199254740992.0);
}
