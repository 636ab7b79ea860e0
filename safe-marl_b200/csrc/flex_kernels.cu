// flex_kernels.cu -- the fused flex_provision kernels (sm_100a).
//
//   k_env<STEP>   replaces FlexibilityProvisionEnv.step           (flexibility_provision_env.py:241-356)
//   k_env<RESET>  replaces reset()/manual_reset()                  (:74-155, :157-239)
//   k_env<PREVIEW> what k_env<STEP> computes for K candidate actions per env, without committing any of it
//   k_power_flow  replaces power_flow_solver_simplified, batched   (utils/pf.py:115-192)
//   k_obs         replaces get_obs() incl. its history side effect (:370-403)
//   k_state       replaces get_state()                             (:358-368)
//   k_stats_fold  folds the per-CTA episode-statistics partials    (madrl/models/model.py:247-265)
//
// Mapping: one warp == one environment, lane k == line k (see flex_common.cuh).  Persistent
// CTAs grid-stride over environments; the topology table is staged into shared memory once
// per CTA; profile rows are read with one coalesced 8-byte load per lane (a 256-byte row per
// warp); everything between those loads and the state write-back stays in registers and
// warp shuffles.  No atomics, no inter-warp communication on the step path.
#include "flex_kernels.cuh"
#include "flex_env_math.cuh"

namespace {

constexpr int WARPS_PER_CTA = FP_CTA_THREADS / 32;
constexpr int SCRATCH_DOUBLES = 32;   // per-warp shared scratch

template <int MODE>
__global__ void __launch_bounds__(FP_CTA_THREADS) k_env(const EnvParams prm) {
    // STEP and PREVIEW (MODE != MODE_RESET) share every stage up to the outputs; a preview walks K N virtual envs
    // v = k N + e, reads the state of env e and the actions of v, and writes outputs of v only
    __shared__ DevTopo s_topo;
    __shared__ double s_scratch[WARPS_PER_CTA][SCRATCH_DOUBLES];
    __shared__ double s_stats[WARPS_PER_CTA][FP_NSTATS];

    stage_topo(&s_topo, prm.topo);
    const DevCfg& c = prm.c;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const LaneTopo lt = load_lane_topo(s_topo, lane);
    const int nl = c.nl, na = c.na;
    const int my_col = s_topo.col[lane];
    const int my_agent = s_topo.agent[lane];               // agent living on this lane's bus
    const int a_col = (lane < na) ? s_topo.agent_col[lane] : 0;
    double* scratch = s_scratch[warp];
    double stat_acc = 0.0;                                 // lane j < FP_NSTATS accumulates stat j

    const int64_t warps_total = (int64_t)gridDim.x * WARPS_PER_CTA;
    const int64_t n_virt = (MODE == MODE_PREVIEW) ? prm.n * prm.pv_k : prm.n;
    for (int64_t v = (int64_t)blockIdx.x * WARPS_PER_CTA + warp; v < n_virt; v += warps_total) {
        const int64_t e = (MODE == MODE_PREVIEW) ? v % prm.n : v;
        if (prm.mask != nullptr && prm.mask[e] == 0) continue;          // warp-uniform

        uint64_t* rec = prm.rec + e * FP_REC_STRIDE;
        // ---------------------------------------------------------------- load per-env record
        int32_t start, steps, hist_n, episode;
        double e_init = 0.0, e_cur = 0.0, cum = 0.0;
        double a0, a1, a2, a3;
        a0 = a1 = a2 = a3 = 0.0;
        if (MODE != MODE_RESET) {
            uint64_t tm = rec[FP_REC_TIME];                              // broadcast load
            start = (int32_t)(uint32_t)tm;
            steps = (int32_t)(tm >> 32);
            if (lane < na) {
                e_init = __longlong_as_double((long long)rec[FP_REC_E_INIT + lane]);
                e_cur = __longlong_as_double((long long)rec[FP_REC_E_CUR + lane]);
                if (prm.act_f64) {
                    const double* a = reinterpret_cast<const double*>(prm.actions) + (v * na + lane) * 4;
                    a0 = a[0]; a1 = a[1]; a2 = a[2]; a3 = a[3];
                } else {
                    // fp32 actions are widened exactly (SURVEY quirk Q6)
                    float4 a = reinterpret_cast<const float4*>(prm.actions)[v * na + lane];
                    a0 = (double)a.x; a1 = (double)a.y; a2 = (double)a.z; a3 = (double)a.w;
                }
            }
            cum = __longlong_as_double((long long)rec[FP_REC_CUM]);
            uint64_t hh = rec[FP_REC_HIST];
            hist_n = (int32_t)(uint32_t)hh;
            episode = (int32_t)(hh >> 32);
        } else {
            uint64_t hh = rec[FP_REC_HIST];
            episode = (int32_t)(hh >> 32);
            hist_n = 0;                                                  // :79-80
            steps = 1;                                                   // :76
            cum = 0.0;                                                   // :77
            if (prm.random) {
                // counter = (global env id lo, hi, episode, block); one Philox block per lane
                const uint64_t gid = (uint64_t)(prm.env_offset + e);
                U4 ctr; ctr.x = (uint32_t)gid; ctr.y = (uint32_t)(gid >> 32); ctr.z = (uint32_t)episode; ctr.w = (uint32_t)lane;
                U4 r = philox4x32_10(ctr, (uint32_t)prm.seed, (uint32_t)(prm.seed >> 32));
                // lane 15: start row; lanes 10..14: E0 of agent lane-10; lanes 0..9 : two actions each
                double u0 = u53(r.x, r.y), u1 = u53(r.z, r.w);
                double lo = 0.9 * (c.e_max / 2), hi = 1.1 * (c.e_max / 2);          // :100
                double e0v = lo + (hi - lo) * u0;
                int32_t st = (int32_t)(u0 * (double)prm.start_range);
                start = __shfl_sync(FULL, st, 15);
                // agent i (lane i) needs actions 4i..4i+3 = blocks (2i, 2i+1)
                double b0 = __shfl_sync(FULL, u0, (2 * lane) & 31), b1 = __shfl_sync(FULL, u1, (2 * lane) & 31);
                double b2 = __shfl_sync(FULL, u0, (2 * lane + 1) & 31), b3 = __shfl_sync(FULL, u1, (2 * lane + 1) & 31);
                double ee = __shfl_sync(FULL, e0v, (10 + lane) & 31);
                if (lane < na) { a0 = b0; a1 = b1; a2 = b2; a3 = b3; e_init = ee; }
            } else {
                start = prm.start[e];
                start = (start < 0) ? 0 : ((start >= prm.start_range) ? prm.start_range - 1 : start);   // a direct C caller's rows stay inside the dataset
                if (lane < na) {
                    e_init = prm.e0[e * na + lane];
                    const double* a = prm.a0 + (e * na + lane) * 4;
                    a0 = a[0]; a1 = a[1]; a2 = a[2]; a3 = a[3];
                }
            }
            e_cur = e_init;                                              // reset clips against E0 (:130)
        }

        // ---------------------------------------------------------------- gather the profile row
        // Quirk Q1: the row in force is max(steps-1, 1); the row loaded after the solve is `steps`.
        const int64_t row = (int64_t)start + ((MODE != MODE_RESET && steps > 1) ? min(steps - 1, c.episode_limit + c.history) : 1);
        double pl = 0.0, ql = 0.0;
        if (lane < nl) {
            pl = __ldg(prm.P + row * nl + my_col);
            ql = __ldg(prm.Q + row * nl + my_col);
        }
        double pv = 0.0, price = 0.0, pload_b = 0.0;
        if (lane < na) {
            pv = __ldg(prm.PVP + row * FP_PVP_STRIDE + lane);
            price = __ldg(prm.PVP + row * FP_PVP_STRIDE + FP_PVP_PRICE);
            pload_b = __ldg(prm.P + row * nl + a_col);
        }

        // ---------------------------------------------------------------- actions -> setpoints
        Setpoint sp; sp.pred = sp.ch = sp.dis = sp.qpv = 0.0;
        double p_bus = 0.0;
        if (lane < na) {
            const bool scale = (MODE == MODE_RESET) || !c.raw_actions;
            sp = apply_actions(c, scale, a0, a1, a2, a3, pload_b, pv, e_cur);
            // net consumption at the building's bus, balance row utils/pf.py:65-75
            p_bus = (((pload_b - sp.pred) - pv) + sp.ch) - sp.dis;
        }
        // hand the building's net injection to the lane that owns its bus
        {
            const int src = (my_agent >= 0) ? my_agent : 0;
            double pb = __shfl_sync(FULL, p_bus, src);
            double qb = __shfl_sync(FULL, sp.qpv, src);
            if (my_agent >= 0) { pl = pb; ql = ql - qb; }               // pf.py:77-83: Qload - Qpv
        }

        // ---------------------------------------------------------------- power flow
        const bool inject = (prm.inject != nullptr) && (prm.inject[e] != 0);
        SweepOut sw = distflow_sweep(lt, pl, ql, lane, c.pf_tol, c.pf_max_iter, inject);

        // ESS update utils/pf.py:96-98 with E_init (quirk Q2) and delta_t
        double e_next = 0.0;
        bool e_bad = false;
        if (lane < na) {
            e_next = e_init + c.delta_t * (c.eta_ch * sp.ch - c.inv_eta_dis * sp.dis);
            e_bad = e_next < c.e_next_lb;                                // E_next in NonNegativeReals (pf.py:46)
            // a NaN action: np.clip keeps it, the reference's NLP gets a NaN injection and its solve raises (:314-337)
            if (MODE != MODE_RESET) e_bad = e_bad || (a0 != a0) || (a1 != a1) || (a2 != a2) || (a3 != a3);
        }
        const bool ok = sw.ok && !__any_sync(FULL, e_bad);              // warp-uniform

        // ---------------------------------------------------------------- voltages, masks
        double V = sqrt(sw.v);                                           // pf.py:108
        double* Vrow = prm.V + e * c.nb;
        if (ok && MODE != MODE_PREVIEW) {
            if (lane < nl) Vrow[my_col + 1] = V;
            if (lane == 0) Vrow[0] = 1.0;                                // slack: sqrt(Vsqr = 1), pf.py:51-53
            if (prm.pfl != nullptr && lane < nl) {
                prm.pfl[e * nl + my_col] = sw.P;
                prm.qfl[e * nl + my_col] = sw.Q;
                prm.isq[e * nl + my_col] = sw.ell;
            }
        } else if (MODE == MODE_STEP || (MODE == MODE_PREVIEW && !ok)) {
            // roll back to the last valid state (:318-328): voltages and setpoints
            if (lane < nl) V = Vrow[my_col + 1];
            if (lane < na) {
                const double* sprow = prm.setp + e * 4 * na;
                sp.pred = sprow[0 * na + lane]; sp.ch = sprow[1 * na + lane];
                sp.dis = sprow[2 * na + lane]; sp.qpv = sprow[3 * na + lane];
            }
        }
        if (MODE == MODE_PREVIEW && prm.pv_V != nullptr) {             // what env.voltages would hold after the step
            double* out = prm.pv_V + v * c.nb;
            if (lane < nl) out[my_col + 1] = V;
            if (lane == 0) out[0] = ok ? 1.0 : Vrow[0];
        }
        const double over = V - c.v_max, under = c.v_min - V;
        const bool viol = (lane < nl) && ((over > 0.0) || (under > 0.0));
        double vterm = 0.0;
        if (viol) vterm = c.voltage_coeff * ((over > under) ? over : under);   // :685 max(0, v-vmax, vmin-v)
        uint32_t vm = __reduce_or_sync(FULL, viol ? (1u << my_col) : 0u);
        const uint64_t vmask = ((uint64_t)vm << 1) | (uint64_t)(c.slack_viol & 1);
        const int vcount = __popc(vm) + (c.slack_viol & 1);
        const bool lviol = (lane < nl) && ok && (sw.ell > s_topo.imax2[lane]);       // utils/opf.py:124-126
        const uint32_t lm = __reduce_or_sync(FULL, lviol ? (1u << my_col) : 0u);

        if (MODE != MODE_RESET) {
            // ------------------------------------------------------------ reward (:679-706)
            double vpen = warp_sum_xor(vterm) + c.slack_pen;
            if (lane < na) {
                scratch[lane * 4 + 0] = price * sp.pred;                          // :681
                scratch[lane * 4 + 1] = c.pv_cost * sp.qpv;                       // :682 (signed, Q4)
                scratch[lane * 4 + 2] = c.ess_cost * (sp.ch + sp.dis);            // :683
                scratch[lane * 4 + 3] = c.discomfort_coeff * (sp.pred * sp.pred); // :684
            }
            __syncwarp();
            if (lane == 0) {
                double rev = scratch[0], der = scratch[1], ess = scratch[2], disc = scratch[3];
                for (int i = 1; i < na; ++i) {                                    // python sum(): left to right
                    rev = rev + scratch[i * 4 + 0];
                    der = der + scratch[i * 4 + 1];
                    ess = ess + scratch[i * 4 + 2];
                    disc = disc + scratch[i * 4 + 3];
                }
                double reward = (((rev - der) - ess) - disc) - vpen;              // :686
                scratch[24 + FP_INFO_REVENUE] = rev;
                scratch[24 + FP_INFO_DER_COST] = der;
                scratch[24 + FP_INFO_ESS_COST] = ess;
                scratch[24 + FP_INFO_DISCOMFORT] = disc;
                scratch[24 + FP_INFO_VOLTAGE_PENALTY] = vpen;
                scratch[24 + FP_INFO_REWARD] = reward;                            // info['reward'] is pre-penalty (:697)
                scratch[24 + FP_INFO_CUMULATIVE] = cum;                           // before adding (:703)
                scratch[24 + FP_INFO_SOLVER_FAILED] = ok ? 0.0 : 1.0;
                if (!ok) reward = reward - c.fail_penalty;                        // :336
                scratch[20] = reward;
                scratch[21] = cum + reward;                                       // :343
            }
            __syncwarp();
            const double reward = scratch[20];
            const int steps_new = steps + 1;                                      // :342
            const bool done = (steps_new >= c.episode_limit) || !ok;              // :345-348
            if (lane < FP_INFO_STRIDE) {
                double iv = scratch[24 + lane];
                if (prm.info != nullptr) prm.info[v * FP_INFO_STRIDE + lane] = iv;
                stat_acc += iv;                     // slots 0..6 info sums, 7 failures
            } else if (lane == 8) stat_acc += (double)vcount;
            else if (lane == 9) stat_acc += 1.0;
            else if (lane == 10) stat_acc += done ? 1.0 : 0.0;
            else if (lane == 11) stat_acc += (double)__popc(lm);
            if (lane == 0) {
                prm.reward[v] = reward;
                prm.done[v] = done ? 1 : 0;
            }
            if (MODE == MODE_PREVIEW) {
                if (lane == 13 && prm.pv_vmask != nullptr) prm.pv_vmask[v] = vmask;
                __syncwarp();                                                     // scratch is reused by the next env
                continue;
            }
            // ------------------------------------------------------------ write back
            // success: E_cur <- E_next; failure: E_cur stays (rolled back). E_init <- E_cur (:354).
            const double e_cur_new = ok ? e_next : e_cur;
            if (lane < na) {
                rec[FP_REC_E_INIT + lane] = (uint64_t)__double_as_longlong(e_cur_new);
                rec[FP_REC_E_CUR + lane] = (uint64_t)__double_as_longlong(e_cur_new);
                if (ok) {
                    double* sprow = prm.setp + e * 4 * na;
                    sprow[0 * na + lane] = sp.pred; sprow[1 * na + lane] = sp.ch;
                    sprow[2 * na + lane] = sp.dis; sprow[3 * na + lane] = sp.qpv;
                }
            }
            if (lane == 10) rec[FP_REC_CUM] = (uint64_t)__double_as_longlong(scratch[21]);
            if (lane == 11) rec[FP_REC_TIME] = pack2(start, steps_new);
            if (lane == 12) rec[FP_REC_HIST] = pack2(hist_n, episode);
            if (lane == 13) rec[FP_REC_VMASK] = vmask;
            if (lane == 14) rec[FP_REC_COUNTS] = pack2(vcount, (done ? FP_FLAG_DONE : 0) | (ok ? 0 : FP_FLAG_FAILED));
            if (lane == 15) rec[FP_REC_LINES] = pack2((int32_t)lm, sw.iters);
            __syncwarp();
        } else {
            // ------------------------------------------------------------ reset write back
            if (lane < na) {
                rec[FP_REC_E_INIT + lane] = (uint64_t)__double_as_longlong(e_init);           // stays E0 (Q2)
                rec[FP_REC_E_CUR + lane] = (uint64_t)__double_as_longlong(ok ? e_next : e_init); // :147
                double* sprow = prm.setp + e * 4 * na;
                sprow[0 * na + lane] = sp.pred; sprow[1 * na + lane] = sp.ch;
                sprow[2 * na + lane] = sp.dis; sprow[3 * na + lane] = sp.qpv;
            }
            if (lane == 10) rec[FP_REC_CUM] = 0;
            if (lane == 11) rec[FP_REC_TIME] = pack2(start, 1);
            if (lane == 12) rec[FP_REC_HIST] = pack2(0, episode + 1);
            if (lane == 13) rec[FP_REC_VMASK] = vmask;
            if (lane == 14) rec[FP_REC_COUNTS] = pack2(vcount, ok ? 0 : FP_FLAG_RESET_FAILED);
            if (lane == 15) rec[FP_REC_LINES] = pack2((int32_t)lm, sw.iters);
        }
    }

    if (MODE == MODE_STEP && prm.stats_partial != nullptr) {
        if (lane < FP_NSTATS) s_stats[warp][lane] = stat_acc;
        __syncthreads();
        if (threadIdx.x < FP_NSTATS) {
            double s = 0.0;
            for (int w = 0; w < WARPS_PER_CTA; ++w) s += s_stats[w][threadIdx.x];
            prm.stats_partial[(int64_t)blockIdx.x * FP_NSTATS + threadIdx.x] += s;   // this CTA owns the row
        }
    }
}

// ------------------------------------------------------------------------ power flow only
__global__ void __launch_bounds__(FP_CTA_THREADS) k_power_flow(const PfParams prm) {
    __shared__ DevTopo s_topo;
    stage_topo(&s_topo, prm.topo);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const LaneTopo lt = load_lane_topo(s_topo, lane);
    const int nl = prm.nl, nb = prm.nl + 1;
    const int my_col = s_topo.col[lane];
    const int64_t warps_total = (int64_t)gridDim.x * WARPS_PER_CTA;
    for (int64_t e = (int64_t)blockIdx.x * WARPS_PER_CTA + warp; e < prm.n; e += warps_total) {
        double p = 0.0, q = 0.0;
        if (lane < nl) {
            p = __ldg(prm.p + e * nl + my_col);
            q = __ldg(prm.q + e * nl + my_col);
        }
        SweepOut sw = distflow_sweep(lt, p, q, lane, prm.tol, prm.max_iter, false);
        if (lane < nl) {
            prm.V[e * nb + my_col + 1] = sqrt(sw.v);
            if (prm.Pl != nullptr) prm.Pl[e * nl + my_col] = sw.P;
            if (prm.Ql != nullptr) prm.Ql[e * nl + my_col] = sw.Q;
            if (prm.Isq != nullptr) prm.Isq[e * nl + my_col] = sw.ell;
        }
        if (lane == 0) {
            prm.V[e * nb] = 1.0;
            if (prm.iters != nullptr) prm.iters[e] = sw.iters;
            if (prm.fail != nullptr) prm.fail[e] = sw.ok ? 0 : 1;
        }
    }
}

// ------------------------------------------------------------------------ observations
// History ring hist[N][H][na][6] fp64 (slot-major: one push is one contiguous 48*na-byte run per env).
// Pushing call k (0-based since reset) writes slot k % H.
template <typename OutT>
__global__ void __launch_bounds__(FP_CTA_THREADS) k_obs(const ObsParams prm) {
    __shared__ double s_cur[WARPS_PER_CTA][32];
    const DevCfg& c = prm.c;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int na = c.na, H = c.history, nl = c.nl;
    const int64_t warps_total = (int64_t)gridDim.x * WARPS_PER_CTA;
    for (int64_t e = (int64_t)blockIdx.x * WARPS_PER_CTA + warp; e < prm.n; e += warps_total) {
        uint64_t* rec = prm.rec + e * FP_REC_STRIDE;
        const uint64_t tm = rec[FP_REC_TIME], hh = rec[FP_REC_HIST];
        const int32_t start = (int32_t)(uint32_t)tm, steps = (int32_t)(tm >> 32);
        const int32_t cnt = (int32_t)(uint32_t)hh;
        const int64_t row = (int64_t)start + ((steps > 1) ? min(steps - 1, c.episode_limit + c.history) : 1);   // row currently loaded (Q1)
        double* hist = prm.hist + e * (int64_t)(H * FP_HIST_SLOT);
        // current 6-vector per agent (:376-384): lanes 0 .. 6*na-1
        const int slot = cnt % H;
        double cur = 0.0;
        if (lane < 6 * na) {
            const int i = lane / 6, f = lane - 6 * i;
            const int col = prm.agent_col[i];
            if (f == 0) cur = __ldg(prm.P + row * nl + col);
            else if (f == 1) cur = __ldg(prm.Q + row * nl + col);
            else if (f == 2) cur = __ldg(prm.PVP + row * FP_PVP_STRIDE + i);
            else if (f == 3) cur = prm.V[e * c.nb + col + 1];
            else if (f == 4) cur = __ldg(prm.PVP + row * FP_PVP_STRIDE + FP_PVP_PRICE);
            else cur = __longlong_as_double((long long)rec[FP_REC_E_CUR + i]);
            if (prm.push) hist[slot * FP_HIST_SLOT + i * 6 + f] = cur;
        }
        s_cur[warp][lane] = cur;
        __syncwarp();
        // window: H entries ending with the current one; entry s (oldest first) is push
        // number (cnt + 1 - H + s); negative -> zero padding (:393-396)
        const int W = H * 6;
        OutT* out = reinterpret_cast<OutT*>(prm.out) + e * (int64_t)(na * W);
        for (int o = lane; o < na * W; o += 32) {
            const int i = o / W, r = o - i * W;
            const int s = r / 6, f = r - 6 * s;
            const int k = cnt + 1 - H + s;                 // push index of this window entry
            double x;
            if (k < 0) x = 0.0;
            else if (k == cnt) x = s_cur[warp][i * 6 + f];
            else x = hist[(k % H) * FP_HIST_SLOT + i * 6 + f];
            out[o] = (OutT)x;
        }
        __syncwarp();
        if (prm.push && lane == 0) rec[FP_REC_HIST] = (hh & 0xffffffff00000000ull) | (uint32_t)(cnt + 1);
    }
}

// Window ring for the rollout loop (one pushing fp32 get_obs per step, model.py:223).
// obsm[N][na][3H][6] fp32: every push writes the agents' 6-vectors ONCE, at slot w (w grows by one per
// push), so the last H entries are the contiguous run of slots w-H+1 .. w and the observation window
// [oldest .. newest] is a strided VIEW of this buffer (agent pitch 3H*6 floats): a push costs 24 bytes
// per agent instead of re-writing the 576-byte row.  When w reaches the end of the ring the last H-1
// entries are copied to its front (k_obsm_compact, once every 2H+1 pushes; the previous view, slots
// 2H .. 3H-1, is not touched by it).  All envs push on every get_obs call, so w is one number for the
// whole batch; a reset zeroes the ring of the envs it resets (k_obsm_clear), which restarts their zero
// padding (:393-396).  The fp64 history ring is still pushed: it stays the source of truth for fp64 /
// non-pushing / out-of-place reads.
__global__ void __launch_bounds__(FP_CTA_THREADS) k_obs_push(const ObsParams prm, float* __restrict__ obsm, int w) {
    const DevCfg& c = prm.c;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int na = c.na, H = c.history;
    const int64_t warps_total = (int64_t)gridDim.x * WARPS_PER_CTA;
    // the record words of the warp's NEXT env are requested before the current env's dependent loads (the kernel is
    // a chain of DRAM round trips: record -> row -> packed observation row)
    int64_t e = (int64_t)blockIdx.x * WARPS_PER_CTA + warp;
    uint64_t tm = 0ull, hh = 0ull;
    if (e < prm.n) { tm = prm.rec[e * FP_REC_STRIDE + FP_REC_TIME]; hh = prm.rec[e * FP_REC_STRIDE + FP_REC_HIST]; }
    for (; e < prm.n; e += warps_total) {
        uint64_t* rec = prm.rec + e * FP_REC_STRIDE;
        const int64_t en = e + warps_total;
        uint64_t tm_next = 0ull, hh_next = 0ull;
        if (en < prm.n) { tm_next = prm.rec[en * FP_REC_STRIDE + FP_REC_TIME]; hh_next = prm.rec[en * FP_REC_STRIDE + FP_REC_HIST]; }
        const int32_t start = (int32_t)(uint32_t)tm, steps = (int32_t)(tm >> 32);
        const int32_t cnt = (int32_t)(uint32_t)hh;
        const int64_t row = (int64_t)start + ((steps > 1) ? min(steps - 1, c.episode_limit + c.history) : 1);   // row currently loaded (Q1)
        // the packed observation row (P, Q at the agent buses, PV, price): one coalesced 128-byte read
        const double orow = (lane < FP_OBS_STRIDE) ? __ldg(prm.OBSROW + row * FP_OBS_STRIDE + lane) : 0.0;
        const int i = lane / 6, f = lane - 6 * i;  // current 6-vector per agent (:376-384): lanes 0 .. 6*na-1
        const int src = (f == 0) ? FP_OBS_P + i : (f == 1) ? FP_OBS_Q + i : (f == 2) ? FP_OBS_PV + i : FP_OBS_PRICE;
        double cur = __shfl_sync(FULL, orow, src & 15);
        if (lane < 6 * na) {
            if (f == 3) cur = prm.V[e * c.nb + prm.agent_col[i] + 1];
            else if (f == 5) cur = __longlong_as_double((long long)rec[FP_REC_E_CUR + i]);
            obsm[(e * na + i) * (int64_t)(3 * H * 6) + w * 6 + f] = (float)cur;
        }
        // the whole warp writes the aligned 256-byte slot (lane = 6 i + f; the pad lanes write zeros): full sectors
        prm.hist[e * (int64_t)(H * FP_HIST_SLOT) + (cnt % H) * FP_HIST_SLOT + lane] = (lane < 6 * na) ? cur : 0.0;
        __syncwarp();
        if (lane == 0) rec[FP_REC_HIST] = (hh & 0xffffffff00000000ull) | (uint32_t)(cnt + 1);
        tm = tm_next; hh = hh_next;
    }
}

// Zero the window ring of the envs a reset touches (mask == nullptr: all): one warp per env, so an
// env that is not reset costs one mask byte.
__global__ void k_obsm_clear(float* __restrict__ obsm, const uint8_t* __restrict__ mask, int64_t n, int per_env) {
    const int lane = threadIdx.x & 31;
    const int64_t warps_total = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t e = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); e < n; e += warps_total) {
        if (mask != nullptr && mask[e] == 0) continue;
        float* wdw = obsm + e * per_env;
        for (int i = lane; i < per_env; i += 32) wdw[i] = 0.f;
    }
}

// End of the ring: copy the last H-1 entries (slots 2H+1 .. 3H-1) of every agent row to slots 0 .. H-2.
__global__ void k_obsm_compact(float* __restrict__ obsm, int64_t rows, int H) {
    // 8-byte pieces: entries are 6 floats, so the row pitch (18 H floats), the source offset ((2 H + 1) * 6) and the
    // run length ((H - 1) * 6) are all even
    const int per = (H - 1) * 3;
    const int64_t total = rows * per;
    float2* o2 = reinterpret_cast<float2*>(obsm);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / per;
        const int k = (int)(i - r * per);
        float2* ring = o2 + r * (int64_t)(3 * H * 3);
        ring[k] = ring[(2 * H + 1) * 3 + k];
    }
}

// Rebuild the window ring from the fp64 history ring (after pushes that went through another path):
// window slot s (oldest first) of every agent lands at ring slot s, i.e. the state after a push at w = H - 1.
__global__ void k_obsm_rebuild(const ObsParams prm, float* __restrict__ obsm) {
    const DevCfg& c = prm.c;
    const int na = c.na, H = c.history;
    const int per_env = na * H * 6;
    const int64_t total = prm.n * (int64_t)per_env;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t e = i / per_env;
        const int r = (int)(i - e * per_env), a = r / (H * 6), r2 = r - a * (H * 6), sl = r2 / 6, f = r2 - 6 * sl;
        const int32_t cnt = (int32_t)(uint32_t)prm.rec[e * FP_REC_STRIDE + FP_REC_HIST];
        const int k = cnt - H + sl;                // push index of window slot sl
        const float x = (k < 0) ? 0.f : (float)prm.hist[e * (int64_t)(H * FP_HIST_SLOT) + (k % H) * FP_HIST_SLOT + a * 6 + f];
        obsm[(e * na + a) * (int64_t)(3 * H * 6) + sl * 6 + f] = x;
    }
}

// ------------------------------------------------------------------------ env-minor observation ring
// The native layout of the observation history for the on-device rollout loop: obsr[H][na][6][n_pad] fp32, n_pad =
// N rounded up to 32.  One push writes, for every (agent, feature), the values of 32 consecutive envs as ONE aligned
// 128-byte line (the env-major window ring writes 24 bytes per agent row: a partial 32-byte sector, which DRAM with ECC
// turns into a read-modify-write), at ring slot q = push number mod H -- one number for the whole batch, because all
// envs push together.  The window of an env is slots q-H+1 .. q (mod H), oldest first; a reset zeroes the env's column,
// which restarts its zero padding (:393-396).  The consumer is the device policy kernel (policy.cu), which reads a
// [144 x 128 envs] block per agent with one TMA box and walks the slots in ring order against permuted weight rows;
// k_obsr_gather materialises the reference's dense [N, na, 6 H] layout for everybody else.
__global__ void k_obsr_rebuild(const ObsParams prm, float* __restrict__ obsr, int64_t n_pad) {
    // from the fp64 history ring (the source of truth): window position s (oldest first) -> ring slot s, i.e. the state
    // after a push at q = H - 1
    const DevCfg& c = prm.c;
    const int na = c.na, H = c.history;
    const int64_t total = (int64_t)H * na * 6 * n_pad;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t rr = i / n_pad, e = i - rr * n_pad;
        const int sl = (int)(rr / (na * 6)), af = (int)(rr - (int64_t)sl * (na * 6));
        float x = 0.f;
        if (e < prm.n) {
            const int32_t cnt = (int32_t)(uint32_t)prm.rec[e * FP_REC_STRIDE + FP_REC_HIST];
            const int k = cnt - H + sl;
            if (k >= 0) x = (float)prm.hist[e * (int64_t)(H * FP_HIST_SLOT) + (k % H) * FP_HIST_SLOT + af];
        }
        obsr[i] = x;
    }
}

// The reverse: restore the fp64 history ring from the env-minor ring after ring-only stepping (fp_set_obs_history(h, 0):
// the fused step then pushes the fp32 ring alone).  Window position s (oldest first) = push number cnt - H + s lives in
// ring slot (q - H + 1 + s) mod H; the restored entries are the fp32 values widened, i.e. every fp32 read of the
// history is unchanged and an fp64 read sees the observation at fp32 precision.
__global__ void k_hist_from_ring(const ObsParams prm, const float* __restrict__ obsr, int64_t n_pad, int q) {
    const DevCfg& c = prm.c;
    const int na = c.na, H = c.history;
    const int64_t total = (int64_t)H * FP_HIST_SLOT * prm.n;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t e = i / (H * FP_HIST_SLOT);
        const int r = (int)(i - e * (H * FP_HIST_SLOT)), s = r / FP_HIST_SLOT, af = r - s * FP_HIST_SLOT;
        const int32_t cnt = (int32_t)(uint32_t)prm.rec[e * FP_REC_STRIDE + FP_REC_HIST];
        const int k = cnt - H + s;
        if (k < 0) continue;
        const int slot = ((q - H + 1 + s) % H + H) % H;
        prm.hist[e * (int64_t)(H * FP_HIST_SLOT) + (k % H) * FP_HIST_SLOT + af] =
            (af < na * 6) ? (double)obsr[((int64_t)slot * na * 6 + af) * n_pad + e] : 0.0;
    }
}

// Zero the columns of the envs a reset touches (mask == nullptr: all).  A thread owns an env: the 32 envs of a warp
// write whole lines when they are reset together (the usual case: episodes of a batch end together).
__global__ void k_obsr_clear(float* __restrict__ obsr, const uint8_t* __restrict__ mask, int64_t n, int64_t n_pad, int rows) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        if (mask != nullptr && mask[e] == 0) continue;
        for (int r = 0; r < rows; ++r) obsr[(int64_t)r * n_pad + e] = 0.f;
    }
}

// The get_obs call at the end of reset() (:155) for the envs a (masked) reset touched, in ring form: the env's column
// is zeroed and its post-reset 6-vectors OVERWRITE the newest slot q -- the terminal observation of the episode that
// just ended, which the rollout loop has consumed -- so that its window reads [0, ..., 0, x_reset] while every other
// env keeps its slot phase (q stays one number for the batch).  Also pushes the fp64 history ring (cnt 0 -> 1).
__global__ void k_obsr_reset_push(const ObsParams prm, float* __restrict__ obsr, int64_t n_pad, int q, const uint8_t* __restrict__ mask) {
    const DevCfg& c = prm.c;
    const int na = c.na, H = c.history;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < prm.n; e += (int64_t)gridDim.x * blockDim.x) {
        if (mask != nullptr && mask[e] == 0) continue;
        uint64_t* rec = prm.rec + e * FP_REC_STRIDE;
        const uint64_t tm = rec[FP_REC_TIME], hh = rec[FP_REC_HIST];
        const int32_t start = (int32_t)(uint32_t)tm, steps = (int32_t)(tm >> 32), cnt = (int32_t)(uint32_t)hh;
        const int64_t row = (int64_t)start + ((steps > 1) ? min(steps - 1, c.episode_limit + c.history) : 1);
        const double* orow = prm.OBSROW + row * FP_OBS_STRIDE;
        double* hslot = prm.hist + e * (int64_t)(H * FP_HIST_SLOT) + (cnt % H) * FP_HIST_SLOT;
        for (int sl = 0; sl < H; ++sl) {
            if (sl == q) continue;
            for (int af = 0; af < na * 6; ++af) obsr[((int64_t)sl * na * 6 + af) * n_pad + e] = 0.f;
        }
        const double price = __ldg(orow + FP_OBS_PRICE);
        for (int i = 0; i < na; ++i) {
            const double x[6] = {__ldg(orow + FP_OBS_P + i), __ldg(orow + FP_OBS_Q + i), __ldg(orow + FP_OBS_PV + i),
                                 prm.V[e * c.nb + prm.agent_col[i] + 1], price, __longlong_as_double((long long)rec[FP_REC_E_CUR + i])};
            for (int f = 0; f < 6; ++f) {
                hslot[i * 6 + f] = x[f];
                obsr[((int64_t)(q * na + i) * 6 + f) * n_pad + e] = (float)x[f];
            }
        }
        for (int k = na * 6; k < FP_HIST_SLOT; ++k) hslot[k] = 0.0;
        rec[FP_REC_HIST] = (hh & 0xffffffff00000000ull) | (uint32_t)(cnt + 1);
    }
}

// Dense view of the ring: out[e][a][s * 6 + f] = obsr[(q - H + 1 + s) mod H][a][f][e]  (the reference's get_obs layout,
// :387-401).  A CTA transposes a tile of (128 envs, one agent) through shared memory -- rows of 129 floats: the row-wise
// fill and the column-wise drain are both conflict-free -- so that both sides move >= 512 contiguous bytes per row (a
// 32-env tile reads 128-byte pieces 512 KB apart, which DRAM serves at less than half its rate).
__global__ void __launch_bounds__(256) k_obsr_gather(const float* __restrict__ obsr, float* __restrict__ out, int64_t n, int64_t n_pad,
                                                     int na, int H, int q) {
    extern __shared__ float tile[];                // [W = 6 H][129]
    const int W = H * 6;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t n_blk = (n + 127) >> 7;
    for (int64_t blk = blockIdx.x; blk < n_blk * na; blk += gridDim.x) {
        const int a = (int)(blk % na);
        const int64_t e0 = (blk / na) << 7;
        for (int k0 = warp; k0 < W; k0 += 32) {    // four rows per warp and trip: sixteen loads in flight per thread
            float v[4][4];
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                const int k = k0 + 8 * m;
                const int sl = k / 6, f = k - 6 * sl;
                int slot = q + 1 + sl; slot = slot >= H ? slot - H : slot;      // q - H + 1 + sl (mod H)
                const float* sp = obsr + ((int64_t)(slot * na + a) * 6 + f) * n_pad + e0 + lane;
#pragma unroll
                for (int i = 0; i < 4; ++i) v[m][i] = (k < W && e0 + lane + 32 * i < n) ? __ldg(sp + 32 * i) : 0.f;
            }
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                const int k = k0 + 8 * m;
                if (k < W) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) tile[k * 129 + lane + 32 * i] = v[m][i];
                }
            }
        }
        __syncthreads();
        for (int j = warp; j < 128; j += 8) {
            if (e0 + j < n) {
                float* dst = out + ((e0 + j) * na + a) * (int64_t)W;
                for (int k = lane; k < W; k += 32) dst[k] = tile[k * 129 + j];
            }
        }
        __syncthreads();
    }
}

template <typename OutT>
__global__ void __launch_bounds__(FP_CTA_THREADS) k_state(const ObsParams prm) {
    const DevCfg& c = prm.c;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int na = c.na, nl = c.nl, nb = c.nb;
    const int W = 3 * nb + 2 * na + 1;
    const int64_t warps_total = (int64_t)gridDim.x * WARPS_PER_CTA;
    // one element of the state vector of env e (row in force `row`): [P(nb) | Q(nb) | Ppv(na) | V(nb) | price | E(na)]
    auto fetch = [&](int64_t e, const uint64_t* rec, int64_t row, int o) -> double {
        int r = o;
        if (r < nb) return (r == 0) ? 0.0 : __ldg(prm.P + row * nl + r - 1);                // :361
        if ((r -= nb) < nb) return (r == 0) ? 0.0 : __ldg(prm.Q + row * nl + r - 1);        // :362
        if ((r -= nb) < na) return __ldg(prm.PVP + row * FP_PVP_STRIDE + r);                // :363
        if ((r -= na) < nb) return prm.V[e * nb + r];                                       // :364
        if ((r -= nb) < 1) return __ldg(prm.PVP + row * FP_PVP_STRIDE + FP_PVP_PRICE);      // :365
        return __longlong_as_double((long long)rec[FP_REC_E_CUR + (r - 1)]);                // :366
    };
    // the (start, step) word of the NEXT env of this warp is requested before the current env's loads, and the
    // four loads a lane owns (W <= 128) are issued together: the kernel is a chain of dependent DRAM round trips
    int64_t e = (int64_t)blockIdx.x * WARPS_PER_CTA + warp;
    uint64_t tm = (e < prm.n) ? prm.rec[e * FP_REC_STRIDE + FP_REC_TIME] : 0ull;
    for (; e < prm.n; e += warps_total) {
        const uint64_t* rec = prm.rec + e * FP_REC_STRIDE;
        const int64_t en = e + warps_total;
        const uint64_t tm_next = (en < prm.n) ? prm.rec[en * FP_REC_STRIDE + FP_REC_TIME] : 0ull;
        const int32_t start = (int32_t)(uint32_t)tm, steps = (int32_t)(tm >> 32);
        const int64_t row = (int64_t)start + ((steps > 1) ? min(steps - 1, c.episode_limit + c.history) : 1);
        OutT* out = reinterpret_cast<OutT*>(prm.out) + e * (int64_t)W;
        double x[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { const int o = lane + 32 * j; x[j] = (o < W) ? fetch(e, rec, row, o) : 0.0; }
#pragma unroll
        for (int j = 0; j < 4; ++j) { const int o = lane + 32 * j; if (o < W) out[o] = (OutT)x[j]; }
        for (int o = lane + 128; o < W; o += 32) out[o] = (OutT)fetch(e, rec, row, o);      // feeders wider than 128 entries
        tm = tm_next;
    }
}

// One warp per statistic: lane l adds rows l, l + 32, ... in order, then a fixed butterfly joins
// the 32 lane sums -- deterministic, and 32 independent load streams instead of one serial chain.
__global__ void k_stats_fold(const double* __restrict__ partial, int n_blocks, double* __restrict__ out) {
    const int j = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (j < FP_NSTATS) {
        double s = 0.0;
        for (int b = lane; b < n_blocks; b += 32) s += partial[(int64_t)b * FP_NSTATS + j];
        s = warp_sum_xor(s);
        if (lane == 0) out[j] = s;
    }
}

// translate_action as a pre-pass (warp / pair variants; the thread kernels fuse it)
__global__ void k_translate_actions(const float* __restrict__ in, float* __restrict__ out, int64_t n, float lo, float hi,
                                    float span) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = translate_action_f32(in[i], lo, hi, span);
}

struct AgentCols { int32_t col[8]; };
__global__ void k_pack_obsrow(const double* __restrict__ P, const double* __restrict__ Q, const double* __restrict__ pvp,
                              const AgentCols ac, int na, int nl, int64_t T, double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= T * FP_OBS_STRIDE) return;
    const int64_t t = i / FP_OBS_STRIDE;
    const int f = (int)(i - t * FP_OBS_STRIDE);
    double x = 0.0;
    if (f < FP_OBS_Q) { if (f < na) x = P[t * nl + ac.col[f]]; }
    else if (f < FP_OBS_PV) { if (f - FP_OBS_Q < na) x = Q[t * nl + ac.col[f - FP_OBS_Q]]; }
    else if (f < FP_OBS_PRICE) { if (f - FP_OBS_PV < na) x = pvp[t * FP_PVP_STRIDE + f - FP_OBS_PV]; }
    else x = pvp[t * FP_PVP_STRIDE + FP_PVP_PRICE];
    out[i] = x;
}

__global__ void k_pack_pvp(const double* __restrict__ pv, const double* __restrict__ price, int na,
                           int64_t T, double* __restrict__ pvp) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= T * FP_PVP_STRIDE) return;
    int64_t t = i / FP_PVP_STRIDE;
    int f = (int)(i - t * FP_PVP_STRIDE);
    double x = 0.0;
    if (f < na) x = pv[t * na + f];
    else if (f == FP_PVP_PRICE) x = price[t];
    pvp[i] = x;
}

}  // namespace

// ------------------------------------------------------------------------ launchers
cudaError_t launch_env(int mode, const EnvParams& prm, int grid, cudaStream_t st) {
    if (mode == MODE_STEP) k_env<MODE_STEP><<<grid, FP_CTA_THREADS, 0, st>>>(prm);
    else if (mode == MODE_PREVIEW) k_env<MODE_PREVIEW><<<grid, FP_CTA_THREADS, 0, st>>>(prm);
    else k_env<MODE_RESET><<<grid, FP_CTA_THREADS, 0, st>>>(prm);
    return cudaGetLastError();
}

cudaError_t launch_power_flow(const PfParams& prm, int grid, cudaStream_t st) {
    k_power_flow<<<grid, FP_CTA_THREADS, 0, st>>>(prm);
    return cudaGetLastError();
}

cudaError_t launch_obs(const ObsParams& prm, int f64, int grid, cudaStream_t st) {
    if (f64) k_obs<double><<<grid, FP_CTA_THREADS, 0, st>>>(prm);
    else k_obs<float><<<grid, FP_CTA_THREADS, 0, st>>>(prm);
    return cudaGetLastError();
}

cudaError_t launch_obs_push(const ObsParams& prm, float* obsm, int q, int grid, cudaStream_t st) {
    k_obs_push<<<grid, FP_CTA_THREADS, 0, st>>>(prm, obsm, q);
    return cudaGetLastError();
}

cudaError_t launch_obsm_clear(float* obsm, const uint8_t* mask, int64_t n, int floats_per_env, cudaStream_t st) {
    const int64_t ctas = (n + 7) / 8;
    k_obsm_clear<<<(unsigned)(ctas < 148 * 8 ? ctas : 148 * 8), 256, 0, st>>>(obsm, mask, n, floats_per_env);
    return cudaGetLastError();
}

cudaError_t launch_obsm_compact(float* obsm, int64_t rows, int H, cudaStream_t st) {
    if (H < 2) return cudaSuccess;
    k_obsm_compact<<<148 * 16, 256, 0, st>>>(obsm, rows, H);
    return cudaGetLastError();
}

cudaError_t launch_obsm_rebuild(const ObsParams& prm, float* obsm, cudaStream_t st) {
    k_obsm_rebuild<<<148 * 16, 256, 0, st>>>(prm, obsm);
    return cudaGetLastError();
}

cudaError_t launch_hist_from_ring(const ObsParams& prm, const float* obsr, int64_t n_pad, int q, cudaStream_t st) {
    k_hist_from_ring<<<148 * 16, 256, 0, st>>>(prm, obsr, n_pad, q);
    return cudaGetLastError();
}
cudaError_t launch_obsr_rebuild(const ObsParams& prm, float* obsr, int64_t n_pad, cudaStream_t st) {
    k_obsr_rebuild<<<148 * 16, 256, 0, st>>>(prm, obsr, n_pad);
    return cudaGetLastError();
}

// Safety layer of SAFEMADDPG (madrl/models/safemaddpg.py:176-299) for every env at once.  The reference builds a QP per
// get_actions call (20 action variables, P_net / Q_net of 33 buses, 66 slacks priced at 1000) and hands it to Gurobi; in
// the form it evaluates the voltage prediction (:266,272: row sums of the coefficient blocks times the bus's OWN P_net /
// Q_net) the problem separates per building into
//     min (x - x0)^2 + (c - c0)^2 + (d - d0)^2 + (g - g0)^2 + w (s_lo + s_up)
//     s.t. V = sP (Pd (1 - x) + c - d) + sQ (Qd + g) + b,  v_min - s_lo <= V <= v_max + s_up,  x, c, d, s >= 0
// whose optimum is closed-form: with a = dV / d(x, c, d, g) pointing towards the violated limit and multiplier
// lam in [0, w], y(lam) = max(y0 + (lam / 2) a, 0) on the bounded variables; the gain a . (y - y0) is concave piecewise
// linear in lam (<= 3 breakpoints, where a decreasing variable reaches zero) and lam* is the smallest multiplier that
// closes the deficit, else w (the rest is slack).  One thread per (env, agent); mirrored by oracle/safety_ref.py.
__global__ void k_safety_project(const SafetyParams prm) {
    const DevCfg& c = prm.o.c;
    const int na = c.na;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < prm.o.n * na; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t e = t / na;
        const int i = (int)(t - e * na);
        // the env's current demands, PV and ESS energy (the row in force, quirk Q1)
        const uint64_t* rec = prm.o.rec + e * FP_REC_STRIDE;
        const int64_t row = row_in_force(c, rec);
        const double* orow = prm.o.OBSROW + row * FP_OBS_STRIDE;
        const double Pd = __ldg(orow + FP_OBS_P + i), Qd = __ldg(orow + FP_OBS_Q + i), ppv = __ldg(orow + FP_OBS_PV + i);
        const double e_cur = __longlong_as_double((long long)rec[FP_REC_E_CUR + i]);
        double a0, a1, a2, a3;
        load_action4(prm.actions, prm.act_f64, t, a0, a1, a2, a3);
        // parse_actions (:143-174) = the env's own scaling / clipping / ESS logic
        const Setpoint sp = apply_actions_frac<true>(c, true, a0, a1, a2, a3, ppv, e_cur);
        double y[4] = {sp.pred, sp.ch, sp.dis, sp.qpv};
        const double sP = prm.sP[i], sQ = prm.sQ[i];
        const double V0 = fma(sQ, Qd + y[3], sP * ((Pd * (1.0 - y[0]) + y[1]) - y[2])) + prm.b[i];
        double slack = 0.0;
        bool moved = false;
        const bool low = V0 < prm.v_min, high = V0 > prm.v_max;
        if (low || high) {
            const double sg = low ? 1.0 : -1.0;
            const double delta = low ? (prm.v_min - V0) : (V0 - prm.v_max);
            const double a[4] = {sg * (-sP * Pd), sg * sP, sg * (-sP), sg * sQ};
            // breakpoints of the bounded variables that move down, sorted (three-element network)
            double bk[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) bk[k] = (a[k] < 0.0) ? (2.0 * y[k] / -a[k]) : prm.w;
            if (bk[0] > bk[1]) { const double s_ = bk[0]; bk[0] = bk[1]; bk[1] = s_; }
            if (bk[1] > bk[2]) { const double s_ = bk[1]; bk[1] = bk[2]; bk[2] = s_; }
            if (bk[0] > bk[1]) { const double s_ = bk[0]; bk[0] = bk[1]; bk[1] = s_; }
            double lam = 0.0, gain = 0.0;
            bool closed = false;
#pragma unroll
            for (int seg = 0; seg < 4 && !closed; ++seg) {
                double nxt = (seg < 3) ? bk[seg] : prm.w;
                nxt = (nxt < prm.w) ? nxt : prm.w;
                if (nxt <= lam) continue;
                double sl = a[3] * a[3] * 0.5;                  // d gain / d lam on (lam, nxt)
#pragma unroll
                for (int k = 0; k < 3; ++k)
                    if (a[k] > 0.0 || (a[k] < 0.0 && lam < 2.0 * y[k] / -a[k])) sl += a[k] * a[k] * 0.5;
                if (sl > 0.0 && gain + sl * (nxt - lam) >= delta) { lam += (delta - gain) / sl; gain = delta; closed = true; }
                else { gain += sl * (nxt - lam); lam = nxt; }
            }
            slack = (delta - gain > 0.0) ? (delta - gain) : 0.0;
#pragma unroll
            for (int k = 0; k < 3; ++k) { const double v = fma(0.5 * lam, a[k], y[k]); y[k] = (v > 0.0) ? v : 0.0; }
            y[3] = fma(0.5 * lam, a[3], y[3]);
            moved = lam > 0.0;
        }
        if (prm.type_major) {
#pragma unroll
            for (int k = 0; k < 4; ++k) prm.out[e * 4 * na + k * na + i] = (float)y[k];    // [x(na) | c(na) | d(na) | g(na)], :290-296
        } else {
            reinterpret_cast<float4*>(prm.out)[t] = make_float4((float)y[0], (float)y[1], (float)y[2], (float)y[3]);
        }
        if (prm.slack != nullptr) prm.slack[t] = slack;
        if (prm.intervened != nullptr) prm.intervened[t] = moved ? 1 : 0;
    }
}
cudaError_t launch_safety_project(const SafetyParams& prm, cudaStream_t st) {
    const int64_t ctas = (prm.o.n * prm.o.c.na + 255) / 256;
    k_safety_project<<<(unsigned)(ctas < 148 * 16 ? ctas : 148 * 16), 256, 0, st>>>(prm);
    return cudaGetLastError();
}

// out[e] = 1 for the envs (of `mask`, if given) whose last reset failed (FP_FLAG_RESET_FAILED); *count = how many
__global__ void k_reset_failed_mask(const uint64_t* __restrict__ rec, const uint8_t* __restrict__ mask, int64_t n,
                                    uint8_t* __restrict__ out, int32_t* __restrict__ count) {
    int local = 0;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t flags = (uint32_t)(rec[e * FP_REC_STRIDE + FP_REC_COUNTS] >> 32);
        const bool bad = ((flags & FP_FLAG_RESET_FAILED) != 0) && (mask == nullptr || mask[e] != 0);
        out[e] = bad ? 1 : 0;
        local += bad ? 1 : 0;
    }
    local = __reduce_add_sync(FULL, local);
    if ((threadIdx.x & 31) == 0 && local) atomicAdd(count, local);
}
cudaError_t launch_reset_failed_mask(const uint64_t* rec, const uint8_t* mask, int64_t n, uint8_t* out, int32_t* count, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(count, 0, 4, st);
    if (e != cudaSuccess) return e;
    const int64_t ctas = (n + 255) / 256;
    k_reset_failed_mask<<<(unsigned)(ctas < 148 * 4 ? ctas : 148 * 4), 256, 0, st>>>(rec, mask, n, out, count);
    return cudaGetLastError();
}

cudaError_t launch_obsr_clear(float* obsr, const uint8_t* mask, int64_t n, int64_t n_pad, int rows, cudaStream_t st) {
    const int64_t ctas = (n + 255) / 256;
    k_obsr_clear<<<(unsigned)(ctas < 148 * 8 ? ctas : 148 * 8), 256, 0, st>>>(obsr, mask, n, n_pad, rows);
    return cudaGetLastError();
}

cudaError_t launch_obsr_reset_push(const ObsParams& prm, float* obsr, int64_t n_pad, int q, const uint8_t* mask, cudaStream_t st) {
    const int64_t ctas = (prm.n + 127) / 128;
    k_obsr_reset_push<<<(unsigned)(ctas < 148 * 16 ? ctas : 148 * 16), 128, 0, st>>>(prm, obsr, n_pad, q, mask);
    return cudaGetLastError();
}

cudaError_t launch_obsr_gather(const float* obsr, float* out, int64_t n, int64_t n_pad, int na, int H, int q, cudaStream_t st) {
    const size_t bytes = (size_t)H * 6 * 129 * sizeof(float);
    if (bytes > 200 * 1024) return cudaErrorInvalidValue;
    cudaError_t e = cudaFuncSetAttribute(k_obsr_gather, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);   // per device: set on every call
    if (e != cudaSuccess) return e;
    const int64_t ctas = ((n + 127) / 128) * na;
    k_obsr_gather<<<(unsigned)(ctas < 148 * 3 ? ctas : 148 * 3), 256, bytes, st>>>(obsr, out, n, n_pad, na, H, q);
    return cudaGetLastError();
}

cudaError_t launch_state(const ObsParams& prm, int f64, int grid, cudaStream_t st) {
    if (f64) k_state<double><<<grid, FP_CTA_THREADS, 0, st>>>(prm);
    else k_state<float><<<grid, FP_CTA_THREADS, 0, st>>>(prm);
    return cudaGetLastError();
}

cudaError_t launch_stats_fold(const double* partial, int n_blocks, double* out, cudaStream_t st) {
    k_stats_fold<<<1, 32 * FP_NSTATS, 0, st>>>(partial, n_blocks, out);
    return cudaGetLastError();
}

cudaError_t launch_pack_obsrow(const double* P, const double* Q, const double* pvp, const int32_t* agent_col, int na, int nl,
                               int64_t T, double* out, cudaStream_t st) {
    AgentCols ac;
    for (int i = 0; i < 8; ++i) ac.col[i] = agent_col[i];
    const int64_t n = T * FP_OBS_STRIDE;
    k_pack_obsrow<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(P, Q, pvp, ac, na, nl, T, out);
    return cudaGetLastError();
}

cudaError_t launch_pack_pvp(const double* pv, const double* price, int na, int64_t T, double* pvp,
                            cudaStream_t st) {
    int64_t n = T * FP_PVP_STRIDE;
    k_pack_pvp<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(pv, price, na, T, pvp);
    return cudaGetLastError();
}

cudaError_t launch_translate_actions(const float* in, float* out, int64_t n, float lo, float hi, float span, cudaStream_t st) {
    k_translate_actions<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(in, out, n, lo, hi, span);
    return cudaGetLastError();
}

int max_resident_grid(int mode) {
    int per_sm = 0, dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaError_t err;
    if (mode == MODE_STEP) err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_env<MODE_STEP>, FP_CTA_THREADS, 0);
    else if (mode == MODE_RESET) err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_env<MODE_RESET>, FP_CTA_THREADS, 0);
    else if (mode == MODE_PREVIEW) err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_env<MODE_PREVIEW>, FP_CTA_THREADS, 0);
    else err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_power_flow, FP_CTA_THREADS, 0);
    if (err != cudaSuccess || per_sm < 1) per_sm = 1;
    return per_sm * sms;
}
