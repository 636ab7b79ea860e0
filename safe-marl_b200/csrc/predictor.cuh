// predictor.cuh -- state of the safety-signal voltage predictor and the device replay ring
// (implemented in predictor.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

// Tile geometry of the tcgen05 predictor kernel: Vhat[128 envs][48] += X[128][72] * A^T[72][48]
#define PRED_M 128          // envs per tile  (UMMA M)
#define PRED_N 48           // outputs padded 33 -> 48 (UMMA N, multiple of 16)
#define PRED_K 72           // inputs padded 66 -> 72 (9 k-steps of 8 tf32)
#define PRED_KC (PRED_K / 4)  // 16-byte chunks along K

struct PredictorState {
    int loaded = 0;
    int n_in = 0, n_out = 0;
    float* d_B = nullptr;      // [2 (hi, lo)][PRED_KC][PRED_N][4] tf32-splittable weights, UMMA K-major layout
    float* d_bias = nullptr;   // [PRED_N]
    double v_min = 0.0, v_max = 0.0, slack_weight = 0.0;
};

void predictor_free(PredictorState* p);

// The MLP of fp_predictor_load_mlp: split weights in the kernel's shared-memory image, padded biases, and the plan.
struct MlpState {
    int loaded = 0;
    float* d_W = nullptr;      // per layer [2 (hi, lo)][k_pad / 4][n_pad][4], UMMA K-major layout
    float* d_bias = nullptr;   // per layer [n_pad]
    int n_layers = 0, act = 0, n_stages = 0, h_cols = 0, n_bias = 0;
    int k_pad[4] = {0, 0, 0, 0}, n_pad[4] = {0, 0, 0, 0}, b_off[4] = {0, 0, 0, 0};
    uint32_t w_off[4] = {0, 0, 0, 0}, w_bytes = 0, smem_bytes = 0;
    double v_min = 0.0, v_max = 0.0, slack_weight = 0.0;
};

void mlp_free(MlpState* m);

struct FpReplay {
    int64_t capacity = 0, head = 0, len = 0;
    int device = 0;
    std::vector<int32_t> widths;
    std::vector<float*> d_fields;      // [capacity][width] each
    std::string err;
};
