/*
 * flexgpu.h -- C ABI of the B200-native batched flex_provision environment.
 *
 * Drop-in boundary for the ONE data-parallel hot path of kosmylo/Safe-MARL: the
 * flex_provision environment step on a radial feeder (IEEE 33-bus), batched over N
 * independent environments that live as device-resident state behind an opaque handle.
 *
 * The reference has no FFI: its boundary is the duck-typed Python MultiAgentEnv API
 * (madrl/environments/multiagentenv.py:1-67) as implemented by
 * madrl/environments/flex_provision/flexibility_provision_env.py.  Each entry point below
 * names the reference function(s) it replaces.  The Python host layer
 * (safe-marl_b200/flexgpu) binds these with ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions
 *   - every function returns 0 on success, a negative FP_E* code otherwise; the message is
 *     available from fp_last_error().  Power-flow non-convergence is NOT an error: it is
 *     reported per environment (flags / info) with the reference's -200 / terminate /
 *     roll-back semantics (flexibility_provision_env.py:314-337).
 *   - pointers named d_* are DEVICE pointers owned by the caller (e.g. torch tensors);
 *     pointers named h_* are HOST pointers.  Nothing is retained after the call returns
 *     except by fp_load_profiles / fp_predictor_load, which copy.
 *   - all work is enqueued on the caller's CUDA stream (`stream` is a cudaStream_t cast
 *     to void*; NULL = legacy default stream).  No entry point synchronises the device
 *     unless it says so.  One handle per GPU per process; a handle is not thread-safe.
 *   - a handle's work runs on the device it was created for, whatever the caller's current
 *     device is: pointers and streams passed with it must belong to that device.  The
 *     caller's current device is unchanged on return.
 *   - there is no CPU fallback: without a CUDA device fp_create fails.
 *
 * Layouts (all row-major, env-major: an env's row is the coalesced unit):
 *   buses are addressed by POSITION in the reference's `bus_numbers` list, slack first
 *   (position 0), as flexibility_provision_env.py:489-490 assumes.  "nl" = n_bus-1 lines;
 *   line k is the line feeding bus position k+1.  "na" = number of agents/buildings.
 */
#ifndef FLEXGPU_H_
#define FLEXGPU_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FP_MAX_BUS     33   /* one lane per line: nl <= 32 */
#define FP_MAX_AGENTS  5
#define FP_INFO_STRIDE 8    /* doubles per env in the info row */
#define FP_NSTATS      16   /* doubles in the episode-statistics vector */

enum {
    FP_OK = 0,
    FP_EINVAL = -1,   /* bad argument / bad topology */
    FP_ECUDA = -2,    /* CUDA runtime error (message has the CUDA string) */
    FP_ESTATE = -3,   /* call sequence error (e.g. step before load_profiles) */
    FP_ENOMEM = -4
};

/* kernel variants (FpConfig.variant).  All compute the same DistFlow fixed point; THREAD and
 * WARP differ in floating-point summation order (results agree to ~1e-12):
 *   THREAD  one CUDA thread per env, one-pass sweep with the currents in registers -- the
 *           throughput path; converges on max_k |P_k^2 + Q_k^2 - v_k l_k| < pf_tol (residual of the
 *           current row, utils/pf.py:85-88, compared on the high words of the fp64 patterns) and
 *           updates the currents once more after the test; default 1e-5 (errors against a Newton
 *           solution: V 1e-11, P/Q 6e-9, I 6e-8 p.u. -- the parity bar is 1e-6).
 *   WARP    one warp per env, lane = line, shuffle scans -- the lowest latency for tiny
 *           batches; converges on max |dv| <= pf_tol (squared voltage), default 1e-9. */
enum { FP_VARIANT_THREAD = 0, FP_VARIANT_WARP = 1 };

/* action dtypes accepted by fp_step */
/* Action dtypes of fp_step / fp_step_host.  FP_F32_POLICY: raw fp32 policy outputs; the kernel
 * applies translate_action (utils/util.py:121-129) itself, in fp32 and in the reference's operation
 * order -- clamp to [action_low, action_high], then 0.5 * (x + 1) * (high - low) + low (quirk Q5) --
 * before widening to fp64, so the rollout loop needs no separate elementwise pass. */
enum { FP_F32 = 0, FP_F64 = 1, FP_F32_POLICY = 2 };

/* info row slots (FP_INFO_STRIDE doubles per env); keys of calculate_reward's dict
 * (flexibility_provision_env.py:696-704) plus the solver_failed flag (:337). */
enum {
    FP_INFO_REWARD = 0, FP_INFO_REVENUE = 1, FP_INFO_DER_COST = 2, FP_INFO_ESS_COST = 3,
    FP_INFO_DISCOMFORT = 4, FP_INFO_VOLTAGE_PENALTY = 5, FP_INFO_CUMULATIVE = 6,
    FP_INFO_SOLVER_FAILED = 7
};

/* flag bits in the per-env record */
enum {
    FP_FLAG_DONE = 1,          /* terminated at the last step (:345-348) */
    FP_FLAG_FAILED = 2,        /* last step's power flow failed (:314-337) */
    FP_FLAG_RESET_FAILED = 4   /* the reset power flow failed; caller must re-draw (:150-153) */
};

/* per-env record: FP_REC_STRIDE 8-byte slots */
#define FP_REC_STRIDE 16
enum {
    FP_REC_E_INIT = 0,     /* [na] double  initial_ess_energy (what the solver sees, quirk Q2) */
    FP_REC_E_CUR = 5,      /* [na] double  current_ess_energy */
    FP_REC_CUM = 10,       /* double       cumulative_reward */
    FP_REC_TIME = 11,      /* int32 start_idx (lo), int32 steps (hi) */
    FP_REC_HIST = 12,      /* int32 obs-history pushes since reset (lo), int32 episode counter (hi) */
    FP_REC_VMASK = 13,     /* uint64 voltage-violation mask, bit b = bus position b */
    FP_REC_COUNTS = 14,    /* int32 violation count (lo), int32 flags (hi) */
    FP_REC_LINES = 15      /* uint32 line-limit mask, bit k = line k (lo), int32 sweep iterations (hi) */
};

/* Configuration = madrl/args/env_args/flex_provision.yaml:3-33 + the topology dict of
 * utils/create_net.py:27-38, already converted to per unit (create_net.py:17-24). */
typedef struct FpConfig {
    int32_t n_bus;               /* len(bus_numbers); slack must be position 0 */
    int32_t n_agents;            /* len(buildings) == len(pv_nodes) == len(ess_nodes) (quirk Q8) */
    int32_t history;             /* yaml history */
    int32_t episode_limit;       /* yaml episode_limit */
    int32_t raw_actions;         /* 1 = 'safemaddpg' branch of step (:268-274): setpoints unscaled */
    int32_t pf_max_iter;         /* sweep iteration cap; exceeding it == solver failure */
    int32_t variant;             /* FP_VARIANT_* */
    int32_t pf_f32_passes;       /* THREAD: opening passes of every solve that run in fp32 (0 = none); the fixed
                                  * point does not depend on how its early iterates were rounded, see DESIGN.md */
    double pf_tol;               /* convergence threshold of the sweep, see FP_VARIANT_* */
    double v_min, v_max;
    double e_min, e_max;
    double p_ch_max, p_dis_max;
    double eta_ch, eta_dis;
    double max_power_reduction;
    double kappa;                /* tan(acos(cos_phi_max)) from the HOST libm (:623) */
    double pv_cost, ess_cost, discomfort_coeff, voltage_coeff;
    double delta_t;              /* 24 / episode_limit (utils/pf.py:23-24) */
    double fail_penalty;         /* 200 (:336) */
    double e_next_lb;            /* E_next lower bound; -1e-8 = IPOPT bound_relax_factor (pf.py:46) */
    int32_t parent[FP_MAX_BUS];  /* parent POSITION of each bus; -1 for the slack */
    double r[FP_MAX_BUS];        /* p.u. resistance of the line feeding bus i (unused for slack) */
    double x[FP_MAX_BUS];
    double imax[FP_MAX_BUS];     /* p.u. rating of that line (max_line_currents) */
    int32_t agent_bus[FP_MAX_AGENTS];  /* bus POSITION of each building */
    int32_t reserved2_[3];
    double action_low, action_high;    /* yaml action_low / action_high: the range translate_action maps into (FP_F32_POLICY) */
} FpConfig;

typedef struct FpHandle FpHandle;

/* -- lifetime ------------------------------------------------------------------------- */

/* Replaces FlexibilityProvisionEnv.__init__ (:34-72) + create_network (create_net.py:8-38)
 * for n_envs environments on CUDA device `device`.  Allocates all per-env state. */
int fp_create(const FpConfig* cfg, int64_t n_envs, int device, FpHandle** out);
int fp_destroy(FpHandle* h);
const char* fp_last_error(const FpHandle* h);   /* h may be NULL: last fp_create error */
int64_t fp_n_envs(const FpHandle* h);

/* Replaces _load_{pv,active_demand,reactive_demand,price}_data (:431-465) after resampling:
 * HOST arrays P[T][nl], Q[T][nl] (non-slack buses, bus order), PV[T][na], price[T].
 * Copies them to the device (synchronous). */
int fp_load_profiles(FpHandle* h, const double* h_P, const double* h_Q, const double* h_PV,
                     const double* h_price, int64_t T);

/* -- episode control -------------------------------------------------------------------- */

/* Replaces reset()/manual_reset() (:74-155, :157-239) for every env whose d_mask byte is
 * non-zero (d_mask == NULL: all).  The caller supplies what the reference draws from
 * np.random (quirk Q9): d_start[N] int32 row of the episode slice (:477), d_e0[N][na]
 * initial ESS energy (:100), d_a0[N][na*4] initial actions (:103), all fp64.
 * Envs whose initial power flow fails get FP_FLAG_RESET_FAILED (the reference re-draws). */
int fp_reset(FpHandle* h, const int32_t* d_start, const double* d_e0, const double* d_a0,
             const uint8_t* d_mask, void* stream);

/* Same, but the draws come from a counter-based Philox4x32-10 stream keyed by
 * (seed, global env id = env_offset + e, per-env episode counter): results do not depend
 * on how envs are sharded over GPUs.  Used by throughput rollouts (auto-reset). */
int fp_reset_random(FpHandle* h, uint64_t seed, int64_t env_offset, const uint8_t* d_mask,
                    void* stream);
/* fp_reset_random, then up to `retries` more launches for the envs (of d_mask) whose initial power flow failed
 * (FP_FLAG_RESET_FAILED) -- the reference's `while not solvable` redraw loop (:82-153) without a host round trip: the
 * retry mask is built on the device.  d_failed (may be NULL): device int32, envs still flagged after the last attempt. */
int fp_reset_random_retry(FpHandle* h, uint64_t seed, int64_t env_offset, const uint8_t* d_mask, int32_t retries,
                          int32_t* d_failed, void* stream);

/* Replaces step() (:241-356): d_actions[N][na*4] (agent-major, k = P_red, P_esc, P_esd, Q_pv)
 * of dtype act_dtype; outputs d_reward[N] fp64, d_done[N] uint8, d_info[N][FP_INFO_STRIDE]
 * fp64 (d_info may be NULL).  d_mask (may be NULL): envs with a zero byte are not stepped
 * (their outputs are left untouched).  A NaN action is a solver failure for its env (np.clip keeps the NaN, the
 * reference's NLP gets a NaN injection and its solve raises, :314-337): roll-back, -200, solver_failed, terminate. */
int fp_step(FpHandle* h, const void* d_actions, int act_dtype, double* d_reward,
            uint8_t* d_done, double* d_info, const uint8_t* d_mask, void* stream);

/* "What would this action do?": what fp_step would compute for k candidate actions per env, bit for bit, WITHOUT
 * committing it.  d_actions[k][N][na*4] of dtype act_dtype (as fp_step, FP_F32_POLICY included); outputs per
 * (candidate, env): d_reward[k][N] fp64, d_done[k][N] uint8, d_info[k][N][FP_INFO_STRIDE] fp64, d_voltage[k][N][n_bus]
 * fp64 (the voltages fp_step would leave behind: after a failed solve, the rolled-back ones), d_vmask[k][N] uint64
 * (the violation mask it would leave in the record); d_info, d_voltage and d_vmask may be NULL.  Candidate c of env e
 * sees env e's current state: the row in force, E_init / E_cur, the episode step and the failure-injection mask of
 * fp_inject_failure.  A failed solve (NaN action included) is reported as fp_step reports it: -200, solver_failed, done.
 * Nothing of the handle is written -- records, voltages, setpoints, line flows, observation history and rings, episode
 * statistics -- so previews may be issued any number of times between two steps, and a step after them gives the
 * same bits as a step without them.  FP_EINVAL for a null actions / reward / done, k < 1 or an unknown dtype;
 * FP_ESTATE before fp_load_profiles. */
int fp_step_preview(FpHandle* h, int32_t k, const void* d_actions, int act_dtype, double* d_reward, uint8_t* d_done,
                    double* d_info, double* d_voltage, uint64_t* d_vmask, void* stream);

/* HOST-buffer variant of fp_step (the end-to-end path): reads h_actions, steps, delivers
 * reward/done/info into the host arrays and synchronises the stream.  h_info may be NULL.
 * With every buffer PINNED (thread variant, FP_F32 or FP_F32_POLICY actions) the step kernel works
 * on them directly (zero-copy: its asynchronous input stage pulls the next tile's actions over PCIe
 * while the current tile is swept, its bulk stores write the results into host memory) -- one
 * launch, no staging.  Otherwise (pageable memory, fp64 actions, warp variant) the actions are
 * copied into device staging buffers, the step runs there and the results are copied back. */
int fp_step_host(FpHandle* h, const void* h_actions, int act_dtype, double* h_reward,
                 uint8_t* h_done, double* h_info, void* stream);

/* -- observations ----------------------------------------------------------------------- */

/* Replaces get_obs() (:370-403): out[N][na][history*6], dtype FP_F32 or FP_F64.
 * push != 0 reproduces the reference's side effect (quirk Q7): the current 6-vector is
 * appended to the per-agent history before the window is read. push == 0 is a pure read
 * of what the next pushing call would return minus the append. */
int fp_get_obs(FpHandle* h, void* d_out, int dtype, int push, void* stream);

/* get_obs() for the rollout loop (one pushing fp32 call per step, madrl/models/model.py:223) WITHOUT
 * re-materialising the window: the handle keeps a window ring [N][na][3*history][6] fp32 into which every
 * push writes the agents' current 6-vectors once, at a slot that advances by one per push, so the last
 * `history` entries are always one contiguous run (at the end of the ring they are copied back to its
 * front, once every 2*history+1 pushes).  push != 0 appends the current 6-vector of every agent (side
 * effect of get_obs, quirk Q7; 24 bytes per agent instead of the whole 576-byte row); *d_view then points
 * at env 0 / agent 0 of the window [oldest .. newest], element (e, i, k) at
 * d_view[e * env_pitch + i * agent_pitch + k], k < history*6, pitches in floats.  The view is read-only for
 * the caller and valid until the next pushing call.  Resets restart the zero padding of the envs they
 * reset.  Pushing through fp_get_obs instead makes the next view call rebuild the ring from the fp64
 * history (correct, one slower call). */
int fp_get_obs_view(FpHandle* h, int push, float** d_view, int64_t* env_pitch, int64_t* agent_pitch, void* stream);

/* fp_step followed by fp_get_obs_view(push = 1) -- the two calls the rollout loop issues every step
 * (madrl/models/model.py:220-223) -- as one entry point (dense view; the one-launch form is fp_step_ring). */
int fp_step_obs(FpHandle* h, const void* d_actions, int act_dtype, double* d_reward, uint8_t* d_done,
                double* d_info, const uint8_t* d_mask, float** d_view, int64_t* env_pitch,
                int64_t* agent_pitch, void* stream);

/* The observation history in its NATIVE device layout, for consumers that stay on the GPU (the policy kernel of the
 * rollout loop, madrl/models/model.py:213-254): an env-minor fp32 ring  ring[history][n_agents][6][n_pad]  (n_pad =
 * n_envs rounded up to 32) in which one pushing get_obs (flexibility_provision_env.py:370-403) writes every
 * (agent, feature) of 32 envs as one aligned 128-byte line at slot `slot` = push number mod history.  The window of
 * an env is slots slot-history+1 .. slot (mod history), oldest first; a reset zeroes its column (the zero padding
 * of :393-396).  Same contents as fp_get_obs; fp_obs_ring_gather materialises the dense [n_envs][n_agents][6 history].
 *   fp_step_ring             fp_step + the pushing get_obs that follows it (model.py:220-223) in ONE launch
 *   fp_obs_ring              the ring as it stands (no push)
 *   fp_obs_ring_reset_push   the get_obs at the end of reset() (:155) for the envs of a masked reset: their column is
 *                            zeroed and the post-reset observation overwrites the newest slot
 *   fp_obs_ring_gather       d_out[n_envs][n_agents][6 history] fp32 = the windows, oldest entry first
 *   fp_set_obs_history       keep = 0: ring-only stepping -- the one-launch fp_step_ring stops maintaining the fp64
 *                            history ring behind fp_get_obs (33 MB of scattered writes per 131 072 envs: 91 -> 79 us per
 *                            step); any later call that needs it (fp_get_obs, fp_get_obs_view, fp_history_ptr) first
 *                            restores it from the ring, i.e. with the history entries at fp32 precision (every fp32
 *                            read is unchanged).  keep = 1 (the default): both rings are pushed */
int fp_step_ring(FpHandle* h, const void* d_actions, int act_dtype, double* d_reward, uint8_t* d_done, double* d_info,
                 const uint8_t* d_mask, float** d_ring, int32_t* slot, int64_t* n_pad, void* stream);
int fp_obs_ring(FpHandle* h, float** d_ring, int32_t* slot, int64_t* n_pad, void* stream);
int fp_obs_ring_reset_push(FpHandle* h, const uint8_t* d_mask, void* stream);
int fp_obs_ring_gather(FpHandle* h, float* d_out, void* stream);
int fp_set_obs_history(FpHandle* h, int keep);

/* Replaces get_state() (:358-368): out[N][2*n_bus + na + n_bus + 1 + na]. */
int fp_get_state(FpHandle* h, void* d_out, int dtype, void* stream);

/* Device pointers to live state (valid until fp_destroy; rows are per env):
 *   rec      uint64/double [N][FP_REC_STRIDE]   (see FP_REC_*)
 *   voltage  double [N][n_bus]                  current_voltage, bus order (:146, :310)
 *   setpoint double [N][4][na]                  power_reduction, ess_charging,
 *                                               ess_discharging, q_pv (:293, :287-290, :281)
 *   pflow/qflow/isq double [N][nl]              receiving-end line flows and squared currents
 *                                               of the last solve (utils/pf.py:109-110); only
 *                                               maintained when fp_set_keep_flows(h, 1)
 *   stats    double [FP_NSTATS]                 see fp_stats_* */
int fp_state_ptrs(FpHandle* h, void** d_rec, void** d_voltage, void** d_setpoint,
                  void** d_pflow, void** d_qflow, void** d_isq);
int fp_set_keep_flows(FpHandle* h, int keep);
/* The fp64 observation-history ring, [N][history][32] doubles (5 x 6 values + 2 pad per entry): with fp_state_ptrs'
 * rec / voltage / setpoint arrays it is the complete per-env device state (checkpointing, SURVEY 5).  write != 0: the
 * caller is about to overwrite it; the derived fp32 observation rings are rebuilt from it on their next use. */
int fp_history_ptr(FpHandle* h, void** d_hist, int64_t* doubles_per_env, int32_t write);

/* -- power flow only (BASELINE config 2) -------------------------------------------------- */

/* Replaces power_flow_solver_simplified (utils/pf.py:115-192), batched: d_p/d_q[N][nl] net
 * consumption of the non-slack buses (bus order) -> d_V[N][n_bus] voltage magnitudes,
 * d_Pl/d_Ql/d_Isq[N][nl] (may be NULL), d_iters[N] int32 (may be NULL), d_fail[N] uint8
 * (may be NULL).  n may differ from the handle's n_envs. */
int fp_power_flow(FpHandle* h, int64_t n, const double* d_p, const double* d_q, double* d_V,
                  double* d_Pl, double* d_Ql, double* d_Isq, int32_t* d_iters, uint8_t* d_fail,
                  void* stream);

/* -- device replay ring (utils/replay_buffer.py:3-30, TransReplayBuffer) ------------------- */

/* A FIFO of `capacity` transitions held as struct-of-arrays fp32 fields on the device
 * (field f: [capacity][widths[f]]).  Head/length bookkeeping lives on the host, so no call
 * synchronises.  Producers reserve rows and write their fields in place (fp_predict does so
 * directly from its epilogue); the learner reads a contiguous window like get_batch. */
typedef struct FpReplay FpReplay;
int fp_replay_create(int64_t capacity, int32_t n_fields, const int32_t* widths, int device, FpReplay** out);
int fp_replay_destroy(FpReplay* r);
const char* fp_replay_last_error(const FpReplay* r);   /* r may be NULL: last fp_replay_create error */
int64_t fp_replay_len(const FpReplay* r);               /* len(self.buffer) */
int64_t fp_replay_capacity(const FpReplay* r);
int fp_replay_clear(FpReplay* r);                       /* clear() (:29-30) */
/* add_experience (:23-27) for n rows at once: returns the ring position of the first row in
 * *pos; when the ring is full the oldest rows are overwritten (offset(), :11-12). */
int fp_replay_reserve(FpReplay* r, int64_t n, int64_t* pos);
/* copy d_src[n][width(field)] into the rows reserved at pos (wraps at capacity) */
int fp_replay_write(FpReplay* r, int32_t field, int64_t pos, int64_t n, const float* d_src, void* stream);
/* get_batch / get_truncated_episodes_batch (:14-21): `batch` CONSECUTIVE rows starting at
 * logical index `start` (0 = oldest; the caller draws start ~ U{0..len-batch} as :18 does).
 * d_out: HOST array of n_fields DEVICE pointers, out[f] = [batch][width(f)]; NULL entries skipped. */
int fp_replay_sample(FpReplay* r, int64_t start, int64_t batch, float* const* d_out, void* stream);
int fp_replay_field_ptr(FpReplay* r, int32_t field, float** d_ptr);

/* -- voltage predictor + safety penalty (BASELINE config 4) ------------------------------- */

/* Replaces the fitted regressor of safety_signal/train_safety_signal_model.py:33-46,73 as an
 * affine map Vhat = A x + c on RAW inputs: the caller folds the MinMax scalers into A [n_out][n_in]
 * and c [n_out] (host, fp64).  x is interleaved [P1,Q1,...,P33,Q33] (data_generation.py:48-50).
 * The safemaddpg row-sum quirk (safemaddpg.py:266,272) is the same map with a 2-banded A.
 * v_min / v_max / slack_weight define the slack penalty of safemaddpg.py:205-229:
 *   penalty = slack_weight * sum_i (max(0, v_min - Vhat_i) + max(0, Vhat_i - v_max)). */
int fp_predictor_load(FpHandle* h, int32_t n_in, int32_t n_out, const double* h_A, const double* h_c,
                      double v_min, double v_max, double slack_weight);
/* Batched inference on tcgen05 tensor cores (3xTF32, fp32 accumulate): d_X [n][66] fp32 (16-byte
 * aligned) -> d_vhat [n][33] fp32 and d_penalty [n] fp64 (either may be NULL).  If sink != NULL the
 * results are ALSO written straight into the replay ring rows pos .. pos+n-1 (mod capacity) of
 * fields f_vhat (width 33) / f_penalty (width 1); a negative field index skips that output. */
int fp_predict(FpHandle* h, int64_t n, const float* d_X, float* d_vhat, double* d_penalty, FpReplay* sink,
               int32_t f_vhat, int32_t f_penalty, int64_t pos, void* stream);

/* The same predictor as a scikit-learn MLPRegressor: 1..3 hidden layers of width 1..128 sharing one activation,
 * identity output layer.  n_layers = hidden layers + 1 (2..4); h_widths[n_layers + 1] = {66, hidden..., 33};
 * h_W = the layers' [out][in] row-major fp64 matrices concatenated, h_b = their biases concatenated (host, copied;
 * the caller folds the MinMax scalers into the first and last layer).  The model is held in its own slot of the
 * handle: loading it does not evict the fp_predictor_load model.  The split-TF32 weights stay in shared memory, so a
 * model is accepted only if they, the output staging and two 33 KB X staging buffers fit the 227 KB of one block, and
 * its TMEM plan fits 512 columns; otherwise, and for bad widths, non-finite weights, an unknown activation,
 * v_min >= v_max or slack_weight <= 0, FP_EINVAL with a message. */
#define FP_ACT_IDENTITY 0
#define FP_ACT_RELU 1
#define FP_ACT_TANH 2
#define FP_ACT_LOGISTIC 3
int fp_predictor_load_mlp(FpHandle* h, int32_t n_layers, const int32_t* h_widths, const double* h_W, const double* h_b,
                          int32_t activation, double v_min, double v_max, double slack_weight);
/* fp_predict's contract (outputs, replay sink, field checks, 16-byte-aligned X) for the model of
 * fp_predictor_load_mlp; FP_ESTATE before it. */
int fp_predict_mlp(FpHandle* h, int64_t n, const float* d_X, float* d_vhat, double* d_penalty, FpReplay* sink,
                   int32_t f_vhat, int32_t f_penalty, int64_t pos, void* stream);

/* -- safety layer as a batched projection (SURVEY 8f rank 4) ------------------------------- */

/* Replaces SAFEMADDPG.safety_layer_optimization (madrl/models/safemaddpg.py:176-299: a Pyomo QP solved by Gurobi per
 * get_actions call) for every env at once.  In the form the reference evaluates its voltage predictor (:266,272: the
 * ROW SUMS of the coefficient blocks coef[:, :33] / coef[:, 33:] times the bus's own P_net / Q_net) the QP separates
 * per building and has a closed-form optimum (k_safety_project).  fp_safety_load takes the fitted regressor as the
 * reference reads it (:182-184): h_coef [n_bus][2 n_bus], h_intercept [n_bus] (host, fp64), the voltage limits and the
 * slack price (1000, :205-206).  fp_safety_project: d_actions [N][na][4] raw policy outputs (FP_F32 / FP_F64) -> parse_actions
 * (:143-174, the env's own scaling / ESS logic on its current demands, PV and energy) -> projection -> d_adjusted fp32,
 * either in the reference's return layout [N][x(na) | c(na) | d(na) | g(na)] (type_major = 1, :290-296) or [N][na][4];
 * d_slack [N][na] (remaining predicted violation, p.u.) and d_intervened [N][na] may be NULL.
 * NaN: parse_actions clips as numpy.clip does, so a NaN action component (or a3 = +-inf where PV = 0, or a1 = a2 = +inf,
 * whose charge / discharge netting is inf - inf) leaves the agent's proposal NaN; it is returned as parsed, with NaN where numpy has it, and not projected: intervened 0, slack 0. */
int fp_safety_load(FpHandle* h, const double* h_coef, const double* h_intercept, double v_min, double v_max, double slack_weight);
int fp_safety_project(FpHandle* h, const void* d_actions, int act_dtype, float* d_adjusted, int32_t type_major, double* d_slack,
                      uint8_t* d_intervened, void* stream);

/* The same layer against the full fitted map as it was trained, V = A [P_1, Q_1, ..., P_nb, Q_nb] + c, instead of the
 * reference's row-sum reading: every bus's prediction depends on every building's actions, so each env solves
 *     min_y sum_k ||y_k - y0_k||^2 + w sum_n [max(0, v_min - V_n(y)) + max(0, V_n(y) - v_max)],  x, c, d >= 0
 * (y0 = parse_actions of the proposal, the injections of safety_ref.solve_reference_qp) by an exact active-set method
 * on the 2 na numbers V depends on (k_safety_project_affine).  The two forms keep separate models.
 * fp_safety_load_affine: h_A [n_out][n_in] and h_c [n_out] (host, fp64: what fp_predictor_load takes) with
 * n_in == 2 n_bus, n_out == n_bus, finite entries, v_min < v_max and slack_weight > 0, else FP_EINVAL.
 * fp_safety_project_affine: inputs and d_adjusted as fp_safety_project; d_slack [N][n_bus] fp64 (remaining predicted
 * violation per bus), d_intervened [N][na] (1 if any of the agent's four values moved) and d_status [N] int32
 * (iterations, 0 if every bus was already inside -- then d_adjusted is the proposal cast to fp32 -- or -1 if the
 * iteration cap was reached) may be NULL.  FP_ESTATE before fp_safety_load_affine or fp_load_profiles.
 * NaN: a proposal that is NaN after parse_actions (as for fp_safety_project) makes V(y0) non-finite, and the whole env
 * is returned as parsed, unprojected: intervened 0 for every agent (the bits did not change), slack 0 on every bus,
 * status 0.  The next fp_step treats the NaN as a solver failure for that env. */
int fp_safety_load_affine(FpHandle* h, int32_t n_in, int32_t n_out, const double* h_A, const double* h_c, double v_min,
                          double v_max, double slack_weight);
int fp_safety_project_affine(FpHandle* h, const void* d_actions, int act_dtype, float* d_adjusted, int32_t type_major,
                             double* d_slack, uint8_t* d_intervened, int32_t* d_status, void* stream);

/* -- acting policy of the rollout loop, transitions, learner feed (SURVEY 8f ranks 1-2) ---- */

/* The shared-parameter RNNAgent (madrl/agents/rnn_agent.py:8-32: fc1(144 obs + na agent-id -> 64) -> LayerNorm ->
 * ReLU -> GRUCell(64) -> fc2(64 -> 4)) evaluated for n_envs x na agents per call on tcgen05 tensor cores, reading the
 * observation ring of fp_step_ring / fp_obs_ring directly, followed by select_action (utils/util.py:50-64, continuous,
 * action_enforcebound) -- i.e. the device form of model.py:215-216 (prep_obs -> get_actions).  Weights are held as
 * TF32; activations keep fp32 accuracy (two-term split).  The handle is independent of FpHandle (one per GPU).
 * na = the handle's agent count, 1 .. 5, fixed for its lifetime (fp_policy_create_agents; fp_policy_create: na = 5).  It
 * must equal the env's n_agents: every shape below is stated with it, and the ring is [24][na][6][n_pad]. */
typedef struct FpPolicy FpPolicy;
int fp_policy_create_agents(int device, int32_t n_agents, FpPolicy** out);   /* FP_EINVAL unless 1 <= n_agents <= 5 */
int fp_policy_create(int device, FpPolicy** out);                            /* = fp_policy_create_agents(device, 5, out) */
int fp_policy_destroy(FpPolicy* p);
const char* fp_policy_last_error(const FpPolicy* p);    /* p may be NULL: last fp_policy_create error */
int64_t fp_policy_launch_count(const FpPolicy* p);
/* HOST fp32 arrays in torch's state_dict layouts: fc1.weight [64][144 + na], fc1.bias [64], layernorm.weight/.bias [64],
 * rnn.weight_ih / weight_hh [192][64] (rows r | z | n), rnn.bias_ih / bias_hh [192], fc2.weight [4][64], fc2.bias [4]. */
int fp_policy_load(FpPolicy* p, const float* fc1_w, const float* fc1_b, const float* ln_g, const float* ln_b,
                   const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh,
                   const float* fc2_w, const float* fc2_b);
/* One acting step.  d_ring / slot / n_pad: the observation ring.  d_hid_in (NULL = zeros) / d_hid_out: hidden states
 * (last_hid / hid of the Transition), [n_envs][na][64] or -- hid_env_minor != 0, the kernel's native layout: every access a
 * coalesced 128-byte line -- [na][64][n_pad] (fp_policy_hidden_to_ring turns it into replay rows); d_reset (may be NULL): envs whose hidden state restarts at zero
 * (init_hidden, model.py:211).  Outputs [n_envs][na][4] fp32: d_mean (may be NULL), d_action = tanh(mean + std eps)
 * (what translate_action receives: feed it to fp_step* with FP_F32_POLICY), d_logp (may be NULL).  explore = 1: status
 * 'train' with exploration, eps from d_eps (caller-supplied standard-normal draws, [n_envs][na][4]) or, if NULL, from
 * Philox4x32-10 keyed by (seed; row, step); explore = 0: status 'test' (action = tanh(mean)).  std = fixed_policy_std. */
int fp_policy_act(FpPolicy* p, const float* d_ring, int32_t slot, int64_t n_pad, int64_t n_envs, const float* d_hid_in,
                  const uint8_t* d_reset, float* d_hid_out, int32_t hid_env_minor, float* d_mean, float* d_action, float* d_logp,
                  const float* d_eps, uint64_t seed, uint64_t step, float std_, int32_t explore, void* stream);
/* select_action alone, on the fc2 outputs a previous fp_policy_act stored in d_mean: another exploration draw of the SAME
 * policy evaluation.  train_process evaluates the policy on (next_state, hid) for the next-value action (model.py:225) and
 * again, on the same inputs, at the top of the next step (:215-216); with this the second evaluation is a re-draw
 * (bit-identical to running fp_policy_act again with these draws). */
int fp_policy_sample(FpPolicy* p, const float* d_mean, int64_t n_envs, float* d_action, float* d_logp, const float* d_eps,
                     uint64_t seed, uint64_t step, float std_, int32_t explore, void* stream);
/* Transition fields (madrl/models/model.py:19, :230-242) straight into a replay ring: field rows (row0 + e) mod cap.
 *   fp_policy_gather_windows   state / next_state: the dense get_obs windows [na][144] of envs [0, n) from the ring
 *                              (pitch = floats per destination row, >= na x 144; row0 = 0, cap >= n: a dense tensor)
 *   fp_policy_hidden_to_ring   last_hid / hid: env-minor hidden states [na][64][n_pad] -> rows of na x 64 floats
 *   fp_policy_rows_to_ring     any dense [n][width] fp32 array (action, log_prob_a, last_hid, hid, value ...)
 *   fp_policy_scalars_to_ring  reward repeated per agent (model.py:221), done, last_step (= done, or every env when
 *                              last_step_all: t == max_steps - 1, model.py:229), all-ones action_avail; NULL fields skipped
 *   fp_policy_transition_tail  ONE launch for all the small fields of a step (model.py:230-242): action, log_prob_a (NULL:
 *                              skipped), reward per agent, done, last_step, action_avail (NULL: skipped) and -- zero_values
 *                              != 0 -- value / next_value as zeros (MADDPG's losses recompute both, maddpg.py:104-107) */
/* One-shot sink for the NEXT fp_policy_act: its writer warps copy the dense get_obs windows of envs [0, n) -- the blocks the
 * kernel stages anyway -- into rows (row0 + e) mod cap of pitch `pitch` floats (>= na x 144; 16-byte aligned field, pitch a multiple of 4):
 * the Transition's `state` without a separate pass over the ring.  Needs n_pad >= 128. */
int fp_policy_state_sink(FpPolicy* p, float* d_field, int64_t pitch, int64_t row0, int64_t cap, int64_t n);
int fp_policy_gather_windows(FpPolicy* p, const float* d_ring, int32_t slot, int64_t n_pad, int64_t n, float* d_out,
                             int64_t pitch, int64_t row0, int64_t cap, void* stream);
int fp_policy_hidden_to_ring(FpPolicy* p, const float* d_hid_em, int64_t n_pad, int64_t n, float* d_field, int64_t row0,
                             int64_t cap, const uint8_t* d_zero_mask, void* stream);
int fp_policy_rows_to_ring(FpPolicy* p, const float* d_src, int64_t n, int32_t width, float* d_field, int64_t row0,
                           int64_t cap, void* stream);
int fp_policy_scalars_to_ring(FpPolicy* p, const double* d_reward, const uint8_t* d_done, int64_t n, int32_t last_step_all,
                              float* f_reward, float* f_done, float* f_last, float* f_avail, int64_t row0, int64_t cap,
                              void* stream);
int fp_policy_transition_tail(FpPolicy* p, const float* d_action, const float* d_logp, const double* d_reward,
                              const uint8_t* d_done, int64_t n, int32_t last_step_all, int32_t zero_values, float* f_action,
                              float* f_logp, float* f_value, float* f_next_value, float* f_reward, float* f_done, float* f_last,
                              float* f_avail, int64_t row0, int64_t cap, void* stream);
/* The critic of the rollout loop: MADDPG.value (madrl/models/maddpg.py:29-76) with the shared-parameter MLPCritic
 * (madrl/critics/mlp_critic.py:5-36: fc1 -> LayerNorm -> ReLU -> fc2 -> ReLU -> fc3) as train_process evaluates it for the
 * Transition's value / next_value (madrl/models/model.py:217, :225-226), on tcgen05 (k_critic), reading the observation
 * ring directly.  fp_critic_load: HOST fp32 arrays in torch's state_dict layouts -- fc1.weight [64][na x 149] (na x 144
 * observation columns | na agent-id columns | na x 4 action columns: 745 for five agents), fc1.bias [64], layernorm.weight
 * / .bias [64], fc2.weight [64][64], fc2.bias [64], fc3.weight [1][64], fc3.bias [1].  fp_critic_value: d_actions
 * [n_envs][na][4] fp32 (what fp_policy_act returned), d_value [n_envs][na] fp32. */
int fp_critic_load(FpPolicy* p, const float* fc1_w, const float* fc1_b, const float* ln_g, const float* ln_b,
                   const float* fc2_w, const float* fc2_b, const float* fc3_w, const float* fc3_b);
int fp_critic_value(FpPolicy* p, const float* d_ring, int32_t slot, int64_t n_pad, int64_t n_envs, const float* d_actions,
                    float* d_value, void* stream);
/* Learner feed: the device part of unpack_data (model.py:308-323) on a batch sampled with fp_replay_sample.
 * d_critic_in [batch * na][na x 149] = the MADDPG critic's input rows (maddpg.py:29-66: all agents' observations, one-hot
 * agent id, all agents' actions; d_state [batch][na x 144], d_action [batch][na x 4]); d_reward [batch][na], d_reward_norm
 * [batch][na] = reward_normalisation (BatchNorm1d over the batch, training
 * mode, initial affine parameters; model.py:321-322).  Either output may be NULL. */
int fp_learner_feed(FpPolicy* p, const float* d_state, const float* d_action, const float* d_reward, int64_t batch,
                    float* d_critic_in, float* d_reward_norm, void* stream);

/* -- episode statistics (the only cross-GPU reduction; madrl/models/model.py:247-265) ----- */

/* Every fp_step adds, per stepped env, to a device vector of FP_NSTATS doubles:
 *   [0..6] sums of the info slots 0..6, [7] solver failures, [8] violation count,
 *   [9] env-steps, [10] episodes finished, [11] line-limit violations, [12..15] reserved.
 * fp_stats_read folds the per-block partials (deterministic order) into d_out[FP_NSTATS];
 * the caller all-reduces d_out across ranks (NCCL) if it shards envs. */
int fp_stats_read(FpHandle* h, double* d_out, void* stream);
int fp_stats_reset(FpHandle* h, void* stream);

/* -- test hooks ------------------------------------------------------------------------- */

/* Fault injection (SURVEY 5): envs whose d_mask byte is non-zero fail their next power
 * flow as if the solver had not converged.  NULL clears. The mask is read at step time. */
int fp_inject_failure(FpHandle* h, const uint8_t* d_mask);

/* Kernel launches issued through this handle since creation (bench's gpu_launches). */
int64_t fp_launch_count(const FpHandle* h);

/* sizeof(FpConfig) as compiled into the library -- lets a foreign-language binding verify
 * its struct layout before the first fp_create. */
int32_t fp_sizeof_config(void);

#ifdef __cplusplus
}
#endif
#endif /* FLEXGPU_H_ */
