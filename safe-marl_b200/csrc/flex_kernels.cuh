// flex_kernels.cuh -- parameter blocks and launcher declarations shared by the kernels
// (flex_kernels.cu) and the C-ABI host layer (flex_api.cu).
#pragma once
#include "flex_common.cuh"

#define FP_CTA_THREADS 256
#define FP_PVP_STRIDE 8        // packed row: PV[0..na-1], price at slot 5, zero padding (64 B)
#define FP_PVP_PRICE 5
#define FP_OBS_STRIDE 16       // packed observation row: P[0..4], Q[5..9] at the agent buses, PV[10..14], price[15]
#define FP_OBS_P 0
#define FP_OBS_Q 5
#define FP_OBS_PV 10
#define FP_OBS_PRICE 15

// MODE_PREVIEW: the step's computation for K candidate actions per env, written to caller buffers; the env's state
// (records, voltages, setpoints, flows, observation rings, statistics) is read and never written (fp_step_preview)
enum { MODE_STEP = 0, MODE_RESET = 1, MODE_PF = 2, MODE_PREVIEW = 3 };

// fp64 history ring: one slot = the agents' 6-vectors (<= 30 doubles) padded to 32 doubles = 256 bytes, so that a
// push writes whole, aligned 32-byte sectors (a partial sector costs a DRAM read-modify-write under ECC)
#define FP_HIST_SLOT 32

struct EnvParams {
    DevCfg c;
    const DevTopo* topo;
    int64_t n;
    // profile dataset (device): P/Q [T][nl] bus order, PVP [T][8]
    const double* P; const double* Q; const double* PVP;
    // thread kernels: the same load rows as (p, q) pairs in DFS lane order, [T][nl][2] -- one
    // contiguous 16*nl-byte row per (env, step), fetched with a single bulk copy
    const double* PQD;
    // what get_obs reads per row, packed: P and Q at the agent buses, PV, price -- one 128-byte row
    const double* OBSROW;
    // fused observation push of step(..., return_obs="ring") (thread kernels): fp64 history ring, env-minor fp32 ring
    // obsr[H][na][6][n_pad], ring slot of this push (obs_push == 0: off)
    double* hist; float* obsr; int64_t n_pad; int32_t obs_push; int32_t obs_q;   // hist: [N][H][FP_HIST_SLOT] doubles
    // per-env state
    uint64_t* rec; double* V; double* setp;
    union {
        struct { double* pfl; double* qfl; double* isq; };          // optional line-flow dump (nullptr = off)
        // MODE_PREVIEW, which never dumps flows: candidates K; per (candidate, env) voltage rows [K][N][nb] and
        // violation masks [K][N] (each may be null).  The actions and reward / done / info are [K][N][...] too.
        struct { double* pv_V; uint64_t* pv_vmask; int64_t pv_k; };
    };
    // step inputs/outputs
    const void* actions; int32_t act_f64;
    // fp32 policy outputs: translate_action (utils/util.py:121-129) in fp32 before widening
    int32_t act_translate; float act_lo, act_hi, act_span;
    double* reward; uint8_t* done; double* info;
    const uint8_t* mask; const uint8_t* inject;
    // reset inputs
    const int32_t* start; const double* e0; const double* a0;
    uint64_t seed; int64_t env_offset; int32_t random; int32_t start_range;
    double* stats_partial;                        // [grid][FP_NSTATS]
    // thread kernels: 32-env tiles [tile_begin, tile_end) of this launch (0, 0 = all, what every launch passes).  Kept:
    // without them ptxas schedules k_env_t differently, and the step measured 0.6 % slower on a B200 (1000 W).
    int64_t tile_begin, tile_end;
    int32_t bulk_io;                              // thread kernels: every per-env output array is 16-byte aligned (bulk stores allowed)
};

struct PfParams {
    const DevTopo* topo;
    int64_t n; int32_t nl; int32_t max_iter; double tol; int32_t n32; int32_t pad_;
    const double* p; const double* q;
    double* V; double* Pl; double* Ql; double* Isq; int32_t* iters; uint8_t* fail;
};

struct ObsParams {
    DevCfg c;
    int64_t n;
    const double* P; const double* Q; const double* PVP;
    const double* OBSROW;                         // [T][16]: P, Q at the agent buses, PV, price (see FP_OBS_*)
    uint64_t* rec; const double* V; double* hist;
    int32_t agent_col[8];
    void* out; int32_t push;
};

// thread-per-env kernels (flex_thread_kernels.cu): same parameter blocks + the by-value topology
struct EnvParamsT { EnvParams e; ThreadTopo t; };
struct PfParamsT { PfParams p; ThreadTopo t; };
enum { VARIANT_THREAD = 0, VARIANT_WARP = 1 };

cudaError_t launch_env_t(int mode, int shape, const EnvParamsT& prm, int grid, cudaStream_t st);
cudaError_t launch_power_flow_t(int shape, const PfParamsT& prm, int grid, cudaStream_t st);
cudaError_t thread_kernels_configure(int n_slots);
cudaError_t launch_pack_pq(const double* P, const double* Q, const ThreadTopo& t, int64_t T, double* pqd, cudaStream_t st);
int thread_kernel_max_grid(int mode, int n_slots, int shape);
int thread_shape_of(const ThreadTopo& t, const int8_t* par_lane);
size_t thread_kernel_smem_bytes(int n_slots);

cudaError_t launch_env(int mode, const EnvParams& prm, int grid, cudaStream_t st);
cudaError_t launch_power_flow(const PfParams& prm, int grid, cudaStream_t st);
cudaError_t launch_obs(const ObsParams& prm, int f64, int grid, cudaStream_t st);
cudaError_t launch_state(const ObsParams& prm, int f64, int grid, cudaStream_t st);
cudaError_t launch_obs_push(const ObsParams& prm, float* obsm, int q, int grid, cudaStream_t st);
cudaError_t launch_obsm_clear(float* obsm, const uint8_t* mask, int64_t n, int floats_per_env, cudaStream_t st);
cudaError_t launch_obsm_rebuild(const ObsParams& prm, float* obsm, cudaStream_t st);
cudaError_t launch_obsm_compact(float* obsm, int64_t rows, int H, cudaStream_t st);
cudaError_t launch_obsr_rebuild(const ObsParams& prm, float* obsr, int64_t n_pad, cudaStream_t st);
cudaError_t launch_hist_from_ring(const ObsParams& prm, const float* obsr, int64_t n_pad, int q, cudaStream_t st);
cudaError_t launch_obsr_clear(float* obsr, const uint8_t* mask, int64_t n, int64_t n_pad, int rows, cudaStream_t st);
cudaError_t launch_obsr_reset_push(const ObsParams& prm, float* obsr, int64_t n_pad, int q, const uint8_t* mask, cudaStream_t st);
cudaError_t launch_obsr_gather(const float* obsr, float* out, int64_t n, int64_t n_pad, int na, int H, int q, cudaStream_t st);
// safety layer of SAFEMADDPG as a batched projection (fp_safety_project)
struct SafetyParams {
    ObsParams o;                                   // c, n, OBSROW, rec (the env's current demands / PV / ESS energy)
    double sP[8], sQ[8], b[8];                     // row sums of the predictor's P / Q coefficient blocks and intercept at the agents' buses
    double v_min, v_max, w;
    const void* actions; int32_t act_f64;          // proposed raw policy actions [n][na][4]
    float* out; int32_t type_major;                // adjusted setpoints: [n][4][na] (the reference's return layout) or [n][na][4]
    double* slack; uint8_t* intervened;            // per (env, agent): remaining slack, 1 if the layer moved the action (may be null)
};
cudaError_t launch_safety_project(const SafetyParams& prm, cudaStream_t st);
// the same layer against the full affine voltage map V = A [P_1, Q_1, ..., P_nb, Q_nb] + c (fp_safety_project_affine)
struct SafetyAffineParams {
    ObsParams o;                                   // c, n, P, Q (full bus rows), OBSROW, rec
    const double* At;                              // the map transposed: At[j * FP_MAX_BUS + n] = A[n][j], j < 2 nb
    const double* cvec;                            // [nb]
    double v_min, v_max, w;
    const void* actions; int32_t act_f64;          // proposed raw policy actions [n][na][4]
    float* out; int32_t type_major;                // adjusted setpoints, layouts as SafetyParams
    double* slack; uint8_t* intervened; int32_t* status;   // [n][nb], [n][na], [n] (each may be null)
};
cudaError_t launch_safety_project_affine(const SafetyAffineParams& prm, cudaStream_t st);

// the profile row in force for env `rec` (quirk Q1): what get_state / the safety layer read as the current demands
__device__ __forceinline__ int64_t row_in_force(const DevCfg& c, const uint64_t* rec) {
    const uint64_t tm = rec[FP_REC_TIME];
    const int32_t start = (int32_t)(uint32_t)tm, steps = (int32_t)(tm >> 32);
    return (int64_t)start + ((steps > 1) ? min(steps - 1, c.episode_limit + c.history) : 1);
}

// raw policy action t (= env * na + agent) of an [n][na][4] fp32 or fp64 array, widened to fp64
__device__ __forceinline__ void load_action4(const void* actions, int32_t act_f64, int64_t t, double& a0, double& a1,
                                             double& a2, double& a3) {
    if (act_f64) {
        const double* ap = reinterpret_cast<const double*>(actions) + t * 4;
        a0 = ap[0]; a1 = ap[1]; a2 = ap[2]; a3 = ap[3];
    } else {
        const float4 f = reinterpret_cast<const float4*>(actions)[t];
        a0 = f.x; a1 = f.y; a2 = f.z; a3 = f.w;
    }
}
cudaError_t launch_reset_failed_mask(const uint64_t* rec, const uint8_t* mask, int64_t n, uint8_t* out, int32_t* count, cudaStream_t st);
cudaError_t launch_stats_fold(const double* partial, int n_blocks, double* out, cudaStream_t st);
cudaError_t launch_pack_obsrow(const double* P, const double* Q, const double* pvp, const int32_t* agent_col, int na, int nl,
                               int64_t T, double* out, cudaStream_t st);
cudaError_t launch_pack_pvp(const double* pv, const double* price, int na, int64_t T, double* pvp,
                            cudaStream_t st);
int max_resident_grid(int mode);

// translate_action (utils/util.py:124-128) on one fp32 action, in the reference's (torch fp32)
// operation order: clamp, + 1, * 0.5, * (high - low), + low.  NaN propagates like th.clamp.
__device__ __forceinline__ float translate_action_f32(float x, float lo, float hi, float span) {
    x = (x < lo) ? lo : ((x > hi) ? hi : x);
    float t = __fadd_rn(x, 1.0f);
    t = __fmul_rn(0.5f, t);
    t = __fmul_rn(t, span);
    return __fadd_rn(t, lo);
}
cudaError_t launch_translate_actions(const float* in, float* out, int64_t n, float lo, float hi, float span, cudaStream_t st);
