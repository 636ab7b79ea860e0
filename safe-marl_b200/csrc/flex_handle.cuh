// flex_handle.cuh -- FpHandle, the per-GPU environment handle of include/flexgpu.h.  Private to the host layers that
// own its entry points: flex_api.cu (environment, safety layer) and predictor.cu (voltage predictor).
#pragma once
#include <cstdint>
#include <string>

#include "flex_kernels.cuh"
#include "predictor.cuh"

struct FpHandle {
    FpConfig cfg;
    DevCfg dc;
    DevTopo topo;
    ThreadTopo tt;               // thread-per-env tables (by-value kernel parameter)
    int variant = FP_VARIANT_THREAD, shape = SHAPE_RUNTIME;
    int64_t n = 0;
    int device = 0;
    int64_t T = 0;
    int32_t start_range = 0;
    // device buffers
    DevTopo* d_topo = nullptr;
    double *d_P = nullptr, *d_Q = nullptr, *d_PVP = nullptr, *d_PQD = nullptr, *d_OBS = nullptr;
    uint64_t* d_rec = nullptr;
    double *d_V = nullptr, *d_setp = nullptr, *d_hist = nullptr;
    // fp32 window ring of the observation history (fp_get_obs_view): [N][na][3H][6], last written slot, validity
    float* d_obsm = nullptr; int obs_q = 0; bool obsm_valid = false;
    // env-minor fp32 ring [H][na][6][n_pad] (fp_step_ring / fp_obs_ring): slot of the newest push, validity
    float* d_obsr = nullptr; int ring_q = 0; bool obsr_valid = false; int64_t n_pad = 0;
    double *d_pfl = nullptr, *d_qfl = nullptr, *d_isq = nullptr;
    double* d_stats_partial = nullptr;
    double safety_sP[8] = {0}, safety_sQ[8] = {0}, safety_b[8] = {0}, safety_vmin = 0, safety_vmax = 0, safety_w = 0; int safety_loaded = 0;
    // the full affine map of fp_safety_load_affine: A transposed [2 nb][FP_MAX_BUS], c [nb]
    double *d_saff_At = nullptr, *d_saff_c = nullptr, saff_vmin = 0, saff_vmax = 0, saff_w = 0; int saff_loaded = 0;
    uint8_t* d_retry_mask = nullptr; void* d_retry_count = nullptr;     // fp_reset_random_retry: device-built retry mask
    int stats_rows = 0;          // rows of the statistics block: the step kernel's grid cap
    const uint8_t* d_inject = nullptr;
    int keep_flows = 0;
    // staging for the host-buffer entry points
    void* d_act_stage = nullptr; double* d_reward_stage = nullptr; uint8_t* d_done_stage = nullptr;
    double* d_info_stage = nullptr;
    float* d_act_xlat = nullptr; int64_t act_xlat_cap = 0;            // FP_F32_POLICY actions translated for the warp kernels
    int cap[4] = {0, 0, 0, 0};   // grid caps of the env kernels by MODE_*: the resident grid, or FLEXGPU_GRID_STEP's below it
    int grid_obs = 0;
    int fuse_obs = 0;            // set around the fp_step of fp_step_obs: the step kernel pushes the observation
    int keep_hist = 1;           // fp_set_obs_history: 0 = the fused ring step does not maintain the fp64 history ring
    bool hist_valid = true;      // false after a ring-only step: restored from the env-minor ring on demand (hist_ensure)
    int64_t launches = 0;
    std::string err;
    PredictorState pred;
    MlpState mlp;                // fp_predictor_load_mlp: its own slot, next to the affine model
};
