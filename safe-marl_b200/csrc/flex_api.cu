// flex_api.cu -- C-ABI host layer of libflexgpu (see include/flexgpu.h).
//
// Owns the per-GPU handle: configuration, the lane-ordered topology tables (the host-side
// equivalent of utils/create_net.py:8-38 plus the DFS pre-order the kernels need), the
// device-resident profile dataset and the per-env state arrays.  No torch types cross this
// boundary; every pointer is a plain host or device pointer.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <new>
#include <cstdint>
#include <string>
#include <vector>

#include "api_handle.cuh"
#include "flex_handle.cuh"

// ------------------------------------------------------------------ topology preprocessing
// Pre-order numbering (children visited in ascending bus position) + per-lane tables.
static int build_topology(const FpConfig& c, DevTopo& t, ThreadTopo& tt, int& shape, std::string& err) {
    const int nb = c.n_bus, nl = nb - 1;
    if (nb < 2 || nb > FP_MAX_BUS) { err = "n_bus must be in [2, 33]"; return FP_EINVAL; }
    if (c.n_agents < 1 || c.n_agents > FP_MAX_AGENTS) { err = "n_agents must be in [1, 5]"; return FP_EINVAL; }
    if (c.parent[0] != -1) { err = "slack bus must be position 0 (parent[0] == -1)"; return FP_EINVAL; }
    std::vector<std::vector<int>> kids(nb);
    for (int b = 1; b < nb; ++b) {
        int p = c.parent[b];
        if (p < 0 || p >= nb || p == b) { err = "parent[] out of range"; return FP_EINVAL; }
        kids[p].push_back(b);                          // ascending b by construction
    }
    std::vector<int> lane_of(nb, -1), bus_of(FP_NL, -1), size(nb, 1);
    // iterative pre-order
    std::vector<int> stack;
    int next = 0;
    for (int i = (int)kids[0].size() - 1; i >= 0; --i) stack.push_back(kids[0][i]);
    std::vector<int> order;
    while (!stack.empty()) {
        int b = stack.back(); stack.pop_back();
        if (lane_of[b] >= 0) { err = "topology has a cycle"; return FP_EINVAL; }
        lane_of[b] = next; bus_of[next] = b; ++next;
        order.push_back(b);
        for (int i = (int)kids[b].size() - 1; i >= 0; --i) stack.push_back(kids[b][i]);
    }
    if (next != nl) { err = "topology is not a connected radial tree rooted at the slack bus"; return FP_EINVAL; }
    for (int i = nl - 1; i >= 0; --i) {                // subtree sizes, children before parents
        int b = order[i];
        if (c.parent[b] != 0) size[c.parent[b]] += size[b];
    }
    std::memset(&t, 0, sizeof(t));
    for (int k = 0; k < FP_NL; ++k) {
        t.end[k] = k; t.col[k] = 0; t.agent[k] = -1;
        t.imax2[k] = std::numeric_limits<double>::infinity();
        uint32_t anc = 0;
        for (int r = 0; r < 5; ++r) anc |= (ANC_NONE << (6 * r));
        t.anc[k] = anc;
    }
    for (int k = 0; k < nl; ++k) {
        int b = bus_of[k];
        if (!(c.r[b] >= 0.0) || !std::isfinite(c.x[b])) { err = "line impedance must be finite"; return FP_EINVAL; }
        t.R[k] = c.r[b]; t.X[k] = c.x[b];
        t.Z2[k] = c.r[b] * c.r[b] + c.x[b] * c.x[b];   // utils/pf.py:93 R**2 + X**2
        t.imax2[k] = (c.imax[b] > 0.0) ? c.imax[b] * c.imax[b] : std::numeric_limits<double>::infinity();
        t.end[k] = k + size[b] - 1;
        t.col[k] = b - 1;
        uint32_t anc = 0;
        for (int r = 0; r < 5; ++r) {
            int a = b;
            for (int s = 0; s < (1 << r) && a > 0; ++s) a = c.parent[a];
            uint32_t al = (a > 0) ? (uint32_t)lane_of[a] : ANC_NONE;
            anc |= (al << (6 * r));
        }
        t.anc[k] = anc;
    }
    for (int i = 0; i < c.n_agents; ++i) {
        int b = c.agent_bus[i];
        if (b < 1 || b >= nb) { err = "agent_bus must be a non-slack bus position"; return FP_EINVAL; }
        if (t.agent[lane_of[b]] >= 0) { err = "two agents on the same bus"; return FP_EINVAL; }
        t.agent[lane_of[b]] = i;
        t.agent_lane[i] = lane_of[b];
        t.agent_col[i] = b - 1;
    }
    // ---- thread-per-env tables: parent lanes -> carry/slot tables (same constexpr derivation
    //      the built-in shapes use at compile time)
    std::memset(&tt, 0, sizeof(tt));
    int8_t par_lane[FP_NL];
    for (int k = 0; k < FP_NL; ++k) par_lane[k] = -1;
    for (int k = 0; k < nl; ++k) {
        int b = bus_of[k];
        par_lane[k] = (int8_t)((c.parent[b] > 0) ? lane_of[c.parent[b]] : -1);
    }
    const TreeTables tb = derive_tree_tables(par_lane, nl);
    bool any_imax = false;
    for (int k = 0; k < FP_NL; ++k) {
        tt.R[k] = t.R[k]; tt.X[k] = t.X[k]; tt.Z2h[k] = 0.5 * t.Z2[k]; tt.imax2[k] = t.imax2[k];
        tt.Rf[k] = (float)tt.R[k]; tt.Xf[k] = (float)tt.X[k]; tt.Z2hf[k] = (float)tt.Z2h[k];
        any_imax = any_imax || (k < nl && std::isfinite(t.imax2[k]));
        tt.par_src[k] = tb.par_src[k]; tt.own_slot[k] = tb.own_slot[k]; tt.dep_slot[k] = tb.dep_slot[k];
        tt.dep_first[k] = tb.dep_first[k]; tt.next_is_child[k] = tb.next_is_child[k];
        tt.chain_of[k] = tb.chain_of[k]; tt.attach_mask[k] = tb.attach_mask[k];
        tt.col[k] = (int8_t)t.col[k];
    }
    for (int c = 0; c < FP_MAX_CHAINS; ++c) tt.child_mask[c] = tb.child_mask[c];
    tt.n_chains = tb.n_chains;
    for (int k = 0; k < nl; ++k) tt.lane_of_col[t.col[k]] = (int8_t)k;
    for (int i = 0; i < 8; ++i) { tt.agent_lane[i] = (int8_t)t.agent_lane[i]; tt.agent_col[i] = (int8_t)t.agent_col[i]; }
    tt.nl = nl; tt.n_slots = tb.n_slots; tt.any_imax = any_imax ? 1 : 0;
    shape = thread_shape_of(tt, par_lane);
    if (c.n_agents != FP_MAX_AGENTS) shape = SHAPE_RUNTIME;      // the built-in shape unrolls the reference's five buildings
    return FP_OK;
}

static void fill_devcfg(const FpConfig& c, DevCfg& d) {
    std::memset(&d, 0, sizeof(d));
    d.nb = c.n_bus; d.nl = c.n_bus - 1; d.na = c.n_agents; d.history = c.history;
    d.episode_limit = c.episode_limit; d.raw_actions = c.raw_actions; d.pf_max_iter = c.pf_max_iter;
    d.obs_w = 6 * c.history;
    d.pf_tol = c.pf_tol; d.v_min = c.v_min; d.v_max = c.v_max; d.e_min = c.e_min; d.e_max = c.e_max;
    d.p_ch_max = c.p_ch_max; d.p_dis_max = c.p_dis_max; d.eta_ch = c.eta_ch; d.eta_dis = c.eta_dis;
    d.inv_eta_ch = 1.0 / c.eta_ch;
    d.inv_eta_dis = 1.0 / c.eta_dis;                   // python evaluates (1 / eta_dis) first (:634, pf.py:97)
    d.mpr = c.max_power_reduction; d.kappa = c.kappa; d.pv_cost = c.pv_cost; d.ess_cost = c.ess_cost;
    d.discomfort_coeff = c.discomfort_coeff; d.voltage_coeff = c.voltage_coeff; d.delta_t = c.delta_t;
    d.fail_penalty = c.fail_penalty; d.e_next_lb = c.e_next_lb;
    // slack bus: V = sqrt(1) = 1 (pf.py:51-53); its penalty term is a constant
    const double over = 1.0 - c.v_max, under = c.v_min - 1.0;
    d.slack_viol = (over > 0.0 || under > 0.0) ? 1 : 0;
    d.slack_pen = d.slack_viol ? c.voltage_coeff * ((over > under) ? over : under) : 0.0;
    d.pf_f32 = c.pf_f32_passes;
}

// envs per CTA of the warp variant's kernels and of the observation kernels: one env per warp
constexpr int64_t ENVS_PER_CTA = FP_CTA_THREADS / 32;

extern "C" {

int fp_create(const FpConfig* cfg, int64_t n_envs, int device, FpHandle** out) {
    if (!cfg || !out || n_envs < 1) return fail<FpHandle>(nullptr, FP_EINVAL, "fp_create: bad arguments");
    if (cfg->history < 1 || cfg->episode_limit < 2 || cfg->pf_max_iter < 1 || !(cfg->pf_tol > 0.0) ||
        cfg->pf_f32_passes < 0 || cfg->pf_f32_passes >= cfg->pf_max_iter ||
        !(cfg->eta_ch > 0.0) || !(cfg->eta_dis > 0.0))
        return fail<FpHandle>(nullptr, FP_EINVAL, "fp_create: bad scalar configuration");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
        return fail<FpHandle>(nullptr, FP_ECUDA, "fp_create: no CUDA device (there is no CPU fallback)");
    if (device < 0 || device >= ndev) return fail<FpHandle>(nullptr, FP_EINVAL, "fp_create: bad device index");
    FpHandle* h = new (std::nothrow) FpHandle();
    if (!h) return fail<FpHandle>(nullptr, FP_ENOMEM, "fp_create: out of host memory");
    h->cfg = *cfg; h->n = n_envs; h->device = device;
    std::string err;
    int rc = build_topology(*cfg, h->topo, h->tt, h->shape, err);
    if (rc != FP_OK) { delete h; return fail<FpHandle>(nullptr, rc, "fp_create: " + err); }
    if (cfg->variant != FP_VARIANT_THREAD && cfg->variant != FP_VARIANT_WARP) {
        delete h; return fail<FpHandle>(nullptr, FP_EINVAL, "fp_create: unknown kernel variant");
    }
    h->variant = cfg->variant;
    if (h->variant == FP_VARIANT_THREAD && (h->tt.n_slots > FP_MAX_SLOTS || h->tt.n_chains > FP_MAX_CHAINS)) {
        delete h; return fail<FpHandle>(nullptr, FP_EINVAL, "fp_create: more than 8 branching buses or 16 laterals; use FP_VARIANT_WARP");
    }
    fill_devcfg(*cfg, h->dc);
    const int nb = cfg->n_bus, na = cfg->n_agents, H = cfg->history;
#define CREATE_TRY(expr)                                                                   \
    do {                                                                                   \
        cudaError_t e_ = (expr);                                                           \
        if (e_ != cudaSuccess) {                                                           \
            std::string m = std::string("fp_create: " #expr ": ") + cudaGetErrorString(e_); \
            fp_destroy(h);                                                                 \
            return fail<FpHandle>(nullptr, e_ == cudaErrorMemoryAllocation ? FP_ENOMEM : FP_ECUDA, m); \
        }                                                                                  \
    } while (0)
    const DeviceGuard on_device(device);
    CREATE_TRY(on_device.error());
    CREATE_TRY(cudaMalloc(&h->d_topo, sizeof(DevTopo)));
    CREATE_TRY(cudaMemcpy(h->d_topo, &h->topo, sizeof(DevTopo), cudaMemcpyHostToDevice));
    CREATE_TRY(cudaMalloc(&h->d_rec, (size_t)n_envs * FP_REC_STRIDE * 8));
    CREATE_TRY(cudaMemset(h->d_rec, 0, (size_t)n_envs * FP_REC_STRIDE * 8));
    CREATE_TRY(cudaMalloc(&h->d_V, (size_t)n_envs * nb * 8));
    CREATE_TRY(cudaMemset(h->d_V, 0, (size_t)n_envs * nb * 8));
    CREATE_TRY(cudaMalloc(&h->d_setp, (size_t)n_envs * 4 * na * 8));
    CREATE_TRY(cudaMemset(h->d_setp, 0, (size_t)n_envs * 4 * na * 8));
    CREATE_TRY(cudaMalloc(&h->d_hist, (size_t)n_envs * H * FP_HIST_SLOT * 8));
    CREATE_TRY(cudaMemset(h->d_hist, 0, (size_t)n_envs * H * FP_HIST_SLOT * 8));
    {   // observation / state kernels are streaming kernels: a full SM worth of warps (8 CTAs of 256 threads)
        int sms = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
        const int64_t ctas = (n_envs + ENVS_PER_CTA - 1) / ENVS_PER_CTA, cap = 8 * (sms > 0 ? sms : 1);
        h->grid_obs = (int)((ctas < cap) ? ctas : cap);
    }
    const bool thread = h->variant == FP_VARIANT_THREAD;
    if (thread) CREATE_TRY(thread_kernels_configure(FP_MAX_SLOTS));
    for (int mode : {MODE_STEP, MODE_RESET, MODE_PF, MODE_PREVIEW})
        h->cap[mode] = thread ? thread_kernel_max_grid(mode, h->tt.n_slots, h->shape) : max_resident_grid(mode);
    h->stats_rows = h->cap[MODE_STEP];
    if (const char* gs = std::getenv("FLEXGPU_GRID_STEP")) {          // tuning knob: persistent CTAs of the thread step kernel
        const int g = std::atoi(gs);
        if (thread && g > 0 && g <= h->cap[MODE_STEP]) h->cap[MODE_STEP] = g;
    }
    CREATE_TRY(cudaMalloc(&h->d_stats_partial, (size_t)h->stats_rows * FP_NSTATS * 8));
    CREATE_TRY(cudaMemset(h->d_stats_partial, 0, (size_t)h->stats_rows * FP_NSTATS * 8));
#undef CREATE_TRY
    *out = h;
    return FP_OK;
}

int fp_destroy(FpHandle* h) {
    if (!h) return FP_OK;
    const DeviceGuard on_device(h->device);       // best effort: the handle is freed whatever happens
    predictor_free(&h->pred);
    mlp_free(&h->mlp);
    cudaFree(h->d_topo); cudaFree(h->d_P); cudaFree(h->d_Q); cudaFree(h->d_PVP); cudaFree(h->d_PQD); cudaFree(h->d_OBS);
    cudaFree(h->d_rec); cudaFree(h->d_V); cudaFree(h->d_setp); cudaFree(h->d_hist); cudaFree(h->d_obsm); cudaFree(h->d_obsr);
    cudaFree(h->d_pfl); cudaFree(h->d_qfl); cudaFree(h->d_isq); cudaFree(h->d_stats_partial); cudaFree(h->d_retry_mask); cudaFree(h->d_retry_count);
    cudaFree(h->d_act_stage); cudaFree(h->d_act_xlat); cudaFree(h->d_reward_stage); cudaFree(h->d_done_stage); cudaFree(h->d_info_stage);
    cudaFree(h->d_saff_At); cudaFree(h->d_saff_c);
    delete h;
    return FP_OK;
}

const char* fp_last_error(const FpHandle* h) { return h ? h->err.c_str() : create_error<FpHandle>().c_str(); }
int64_t fp_n_envs(const FpHandle* h) { return h ? h->n : 0; }
int64_t fp_launch_count(const FpHandle* h) { return h ? h->launches : 0; }
int32_t fp_sizeof_config(void) { return (int32_t)sizeof(FpConfig); }

int fp_load_profiles(FpHandle* h, const double* h_P, const double* h_Q, const double* h_PV,
                     const double* h_price, int64_t T) {
    if (!h) return FP_EINVAL;
    if (!h_P || !h_Q || !h_PV || !h_price) return fail(h, FP_EINVAL, "fp_load_profiles: null array");
    const int nl = h->dc.nl, na = h->dc.na;
    // the reference slices episode_limit + history + 1 rows per episode (:478)
    const int64_t need = (int64_t)h->cfg.episode_limit + h->cfg.history + 1;
    if (T < need) return fail(h, FP_EINVAL, "fp_load_profiles: fewer rows than one episode slice");
    USE_DEVICE(h);
    cudaFree(h->d_P); cudaFree(h->d_Q); cudaFree(h->d_PVP); cudaFree(h->d_PQD); cudaFree(h->d_OBS);
    h->d_P = h->d_Q = h->d_PVP = h->d_PQD = h->d_OBS = nullptr;
    double *d_pv = nullptr, *d_price = nullptr;
    CUDA_TRY(h, cudaMalloc(&h->d_P, (size_t)T * nl * 8));
    CUDA_TRY(h, cudaMalloc(&h->d_Q, (size_t)T * nl * 8));
    CUDA_TRY(h, cudaMalloc(&h->d_PVP, (size_t)T * FP_PVP_STRIDE * 8));
    CUDA_TRY(h, cudaMalloc(&d_pv, (size_t)T * na * 8));
    CUDA_TRY(h, cudaMalloc(&d_price, (size_t)T * 8));
    CUDA_TRY(h, cudaMemcpy(h->d_P, h_P, (size_t)T * nl * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->d_Q, h_Q, (size_t)T * nl * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(d_pv, h_PV, (size_t)T * na * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(d_price, h_price, (size_t)T * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(h, launch_pack_pvp(d_pv, d_price, na, T, h->d_PVP, 0));
    h->launches++;
    CUDA_TRY(h, cudaMalloc(&h->d_OBS, (size_t)T * FP_OBS_STRIDE * 8));
    CUDA_TRY(h, launch_pack_obsrow(h->d_P, h->d_Q, h->d_PVP, h->topo.agent_col, na, nl, T, h->d_OBS, 0));
    h->launches++;
    if (h->variant == FP_VARIANT_THREAD) {   // (p, q) pairs in DFS lane order for the thread kernels
        CUDA_TRY(h, cudaMalloc(&h->d_PQD, (size_t)T * nl * 16));
        CUDA_TRY(h, launch_pack_pq(h->d_P, h->d_Q, h->tt, T, h->d_PQD, 0));
        h->launches++;
    }
    CUDA_TRY(h, cudaDeviceSynchronize());
    cudaFree(d_pv); cudaFree(d_price);
    h->T = T;
    h->start_range = (int32_t)((T - need + 1 < 2147483647LL) ? (T - need + 1) : 2147483647LL);
    return FP_OK;
}

static void fill_env_params(FpHandle* h, EnvParams& p) {
    std::memset(&p, 0, sizeof(p));
    p.c = h->dc; p.topo = h->d_topo; p.n = h->n;
    p.P = h->d_P; p.Q = h->d_Q; p.PVP = h->d_PVP; p.PQD = h->d_PQD; p.OBSROW = h->d_OBS;
    p.rec = h->d_rec; p.V = h->d_V; p.setp = h->d_setp;
    if (h->keep_flows) { p.pfl = h->d_pfl; p.qfl = h->d_qfl; p.isq = h->d_isq; }
    p.inject = h->d_inject;
    p.start_range = h->start_range;
}

// whole-tile bulk stores (thread kernels) need 16-byte aligned output arrays
static int bulk_io_ok(const EnvParams& p) {
    auto al16 = [](const void* x) { return (reinterpret_cast<uintptr_t>(x) & 15u) == 0; };
    return (al16(p.rec) && al16(p.setp) && al16(p.V) && al16(p.reward) && al16(p.done) && (p.info == nullptr || al16(p.info))) ? 1 : 0;
}

// The env kernel of `mode` on the handle's variant, over k candidates per env for MODE_PREVIEW (k = 1 otherwise), on
// at most its resident grid.  translate: p.actions are raw fp32 policy outputs (FP_F32_POLICY), translated into the
// step kernel (thread variant) or by an elementwise pre-pass into the handle's scratch (warp variant).
static int launch_env_any(FpHandle* h, int mode, EnvParams p, bool translate, int64_t k, cudaStream_t st) {
    // translate_action's constants exactly as torch forms them (utils/util.py:124-128): the clamp bounds
    // and `low` become fp32 scalars, `high - low` is a Python (double) difference turned into an fp32 scalar
    const float lo = (float)h->cfg.action_low, hi = (float)h->cfg.action_high;
    const float span = (float)(h->cfg.action_high - h->cfg.action_low);
    const int cap = h->cap[mode];
    if (h->variant == FP_VARIANT_THREAD) {
        EnvParamsT pt;
        pt.e = p; pt.t = h->tt;
        if (translate) { pt.e.act_translate = 1; pt.e.act_lo = lo; pt.e.act_hi = hi; pt.e.act_span = span; }
        if (mode == MODE_STEP) pt.e.bulk_io = bulk_io_ok(p);
        const int64_t tiles = k * ((h->n + 31) / 32);           // 32-env tiles; every candidate's envs start a tile
        CUDA_TRY(h, launch_env_t(mode, h->shape, pt, (int)((tiles < cap) ? tiles : cap), st));
    } else {
        if (translate) {
            const int64_t cnt = k * h->n * h->dc.na * 4;
            if (cnt > h->act_xlat_cap) {
                cudaFree(h->d_act_xlat); h->d_act_xlat = nullptr; h->act_xlat_cap = 0;
                CUDA_TRY(h, cudaMalloc(&h->d_act_xlat, (size_t)cnt * 4));
                h->act_xlat_cap = cnt;
            }
            CUDA_TRY(h, launch_translate_actions((const float*)p.actions, h->d_act_xlat, cnt, lo, hi, span, st));
            h->launches++;
            p.actions = h->d_act_xlat;
        }
        const int64_t ctas = (k * h->n + ENVS_PER_CTA - 1) / ENVS_PER_CTA;
        CUDA_TRY(h, launch_env(mode, p, (int)((ctas < cap) ? ctas : cap), st));
    }
    h->launches++;
    return FP_OK;
}

// Restarts the observation rings of the envs of d_mask (all envs: null) after their reset: the zero padding of their
// windows in the window ring, their history in the env-minor ring.  A ring that is not valid is rebuilt on its next use.
static int restart_obs_rings(FpHandle* h, const uint8_t* d_mask, cudaStream_t st) {
    if (h->d_obsm && h->obsm_valid) {
        CUDA_TRY(h, launch_obsm_clear(h->d_obsm, d_mask, h->n, h->dc.na * 3 * h->dc.history * 6, st));
        h->launches++;
    }
    if (h->d_obsr && h->obsr_valid) {
        CUDA_TRY(h, launch_obsr_clear(h->d_obsr, d_mask, h->n, h->n_pad, h->dc.history * h->dc.na * 6, st));
        h->launches++;
    }
    return FP_OK;
}

// The preamble of the entry points that need the profile dataset: a handle, its device current for the rest of the
// call, profiles loaded.  `what` is the entry point's name, a string literal.
#define ENV_ENTRY(h, what)                                                                                \
    if (!(h)) return FP_EINVAL;                                                                           \
    USE_DEVICE(h);                                                                                        \
    if (!(h)->d_P) return fail((h), FP_ESTATE, what ": call fp_load_profiles first")

// The action dtypes of the stepping entry points
static bool step_dtype_ok(int act_dtype) { return act_dtype == FP_F32 || act_dtype == FP_F64 || act_dtype == FP_F32_POLICY; }

int fp_reset(FpHandle* h, const int32_t* d_start, const double* d_e0, const double* d_a0,
             const uint8_t* d_mask, void* stream) {
    ENV_ENTRY(h, "fp_reset");
    if (!d_start || !d_e0 || !d_a0) return fail(h, FP_EINVAL, "fp_reset: null input");
    EnvParams p; fill_env_params(h, p);
    p.start = d_start; p.e0 = d_e0; p.a0 = d_a0; p.mask = d_mask; p.random = 0;
    p.inject = nullptr;
    const int rc = launch_env_any(h, MODE_RESET, p, false, 1, (cudaStream_t)stream);
    return (rc != FP_OK) ? rc : restart_obs_rings(h, d_mask, (cudaStream_t)stream);
}

// One launch of the random reset for the envs of d_mask (+ the observation rings' restart).
static int reset_random_once(FpHandle* h, uint64_t seed, int64_t env_offset, const uint8_t* d_mask, void* stream) {
    EnvParams p; fill_env_params(h, p);
    p.mask = d_mask; p.random = 1; p.seed = seed; p.env_offset = env_offset;
    p.inject = nullptr;
    const int rc = launch_env_any(h, MODE_RESET, p, false, 1, (cudaStream_t)stream);
    return (rc != FP_OK) ? rc : restart_obs_rings(h, d_mask, (cudaStream_t)stream);
}

int fp_reset_random(FpHandle* h, uint64_t seed, int64_t env_offset, const uint8_t* d_mask, void* stream) {
    ENV_ENTRY(h, "fp_reset_random");
    return reset_random_once(h, seed, env_offset, d_mask, stream);
}

// The reference redraws until the initial power flow is solvable (`while not solvable`, :82-153).  Here: the random
// reset, then `retries` more launches for the envs (of d_mask) whose FP_FLAG_RESET_FAILED is set -- the retry mask is
// built on the device, so nothing synchronises with the host; a launch whose mask is empty costs a few microseconds.
// Every attempt draws from the env's next Philox episode counter.  d_failed (may be NULL) receives the number of envs
// still flagged after the last attempt (int32 on the device).
int fp_reset_random_retry(FpHandle* h, uint64_t seed, int64_t env_offset, const uint8_t* d_mask, int32_t retries,
                          int32_t* d_failed, void* stream) {
    ENV_ENTRY(h, "fp_reset_random_retry");
    if (retries < 0 || retries > 64) return fail(h, FP_EINVAL, "fp_reset_random_retry: 0 <= retries <= 64");
    int rc = reset_random_once(h, seed, env_offset, d_mask, stream);
    if (rc != FP_OK) return rc;
    if (retries > 0 || d_failed) {
        if (!h->d_retry_mask) CUDA_TRY(h, cudaMalloc(&h->d_retry_mask, (size_t)h->n + 4));
        int32_t* cnt = reinterpret_cast<int32_t*>(h->d_retry_count);
        if (!cnt) { CUDA_TRY(h, cudaMalloc(&h->d_retry_count, 4)); cnt = reinterpret_cast<int32_t*>(h->d_retry_count); }
        for (int r = 0; r <= retries; ++r) {
            CUDA_TRY(h, launch_reset_failed_mask(h->d_rec, d_mask, h->n, h->d_retry_mask, cnt, (cudaStream_t)stream));
            h->launches++;
            if (r == retries) break;
            rc = reset_random_once(h, seed, env_offset, h->d_retry_mask, stream);
            if (rc != FP_OK) return rc;
        }
        if (d_failed) CUDA_TRY(h, cudaMemcpyAsync(d_failed, cnt, 4, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    }
    return FP_OK;
}

int fp_step(FpHandle* h, const void* d_actions, int act_dtype, double* d_reward, uint8_t* d_done,
            double* d_info, const uint8_t* d_mask, void* stream) {
    ENV_ENTRY(h, "fp_step");
    if (!d_actions || !d_reward || !d_done) return fail(h, FP_EINVAL, "fp_step: null input/output");
    if (!step_dtype_ok(act_dtype)) return fail(h, FP_EINVAL, "fp_step: bad action dtype");
    EnvParams p; fill_env_params(h, p);
    p.actions = d_actions; p.act_f64 = (act_dtype == FP_F64);
    p.reward = d_reward; p.done = d_done; p.info = d_info; p.mask = d_mask;
    p.stats_partial = h->d_stats_partial;
    if (h->fuse_obs) { p.obs_push = 1; p.obs_q = h->ring_q; p.hist = h->keep_hist ? h->d_hist : nullptr; p.obsr = h->d_obsr; p.n_pad = h->n_pad; }
    return launch_env_any(h, MODE_STEP, p, act_dtype == FP_F32_POLICY, 1, (cudaStream_t)stream);
}

// The step's computation for k candidate actions per env, without committing it: one launch of the step kernel's
// MODE_PREVIEW instantiation over k N virtual envs (see k_env_t).  It reads the handle's state and writes only the
// caller's buffers, so any number of previews may run between two steps.
int fp_step_preview(FpHandle* h, int32_t k, const void* d_actions, int act_dtype, double* d_reward, uint8_t* d_done,
                    double* d_info, double* d_voltage, uint64_t* d_vmask, void* stream) {
    ENV_ENTRY(h, "fp_step_preview");
    if (!d_actions || !d_reward || !d_done) return fail(h, FP_EINVAL, "fp_step_preview: null input/output");
    if (k < 1) return fail(h, FP_EINVAL, "fp_step_preview: k must be >= 1");
    if (!step_dtype_ok(act_dtype)) return fail(h, FP_EINVAL, "fp_step_preview: bad action dtype");
    EnvParams p; fill_env_params(h, p);
    p.pv_V = d_voltage; p.pv_vmask = d_vmask; p.pv_k = k;            // (replaces the line-flow dump, which a preview never writes)
    p.actions = d_actions; p.act_f64 = (act_dtype == FP_F64);
    p.reward = d_reward; p.done = d_done; p.info = d_info;
    return launch_env_any(h, MODE_PREVIEW, p, act_dtype == FP_F32_POLICY, k, (cudaStream_t)stream);
}

// Host-buffer step, on one of two routes chosen from the call itself:
//  * zero-copy (thread variant, every buffer pinned, fp32 actions): pinned host memory is part of the unified
//    address space, so the step kernel reads the actions of tile i+1 straight over PCIe while it sweeps tile i (its
//    input stage is asynchronous and one tile ahead) and stores reward / done / info straight into the host
//    buffers -- one launch, no staging.  fp64 actions are read with plain loads, not LDGSTS, so they are staged.
//  * staged, everything else: one copy in, the step on the device staging buffers, the copies out.
int fp_step_host(FpHandle* h, const void* h_actions, int act_dtype, double* h_reward, uint8_t* h_done,
                 double* h_info, void* stream) {
    ENV_ENTRY(h, "fp_step_host");
    if (!h_actions || !h_reward || !h_done) return fail(h, FP_EINVAL, "fp_step_host: null buffer");
    if (!step_dtype_ok(act_dtype)) return fail(h, FP_EINVAL, "fp_step_host: bad action dtype");
    cudaStream_t st = (cudaStream_t)stream;
    auto pinned = [](const void* x) {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, x) != cudaSuccess) { cudaGetLastError(); return false; }
        return at.type == cudaMemoryTypeHost;
    };
    if (h->variant == FP_VARIANT_THREAD && act_dtype != FP_F64 &&
        pinned(h_actions) && pinned(h_reward) && pinned(h_done) && (!h_info || pinned(h_info))) {
        int rc = fp_step(h, h_actions, act_dtype, h_reward, h_done, h_info, nullptr, stream);
        if (rc != FP_OK) return rc;
    } else {
        const size_t n = (size_t)h->n, na = (size_t)h->dc.na;
        if (!h->d_act_stage)
            CUDA_TRY(h, alloc_group({{&h->d_act_stage, n * na * 4 * 8}, {&h->d_reward_stage, n * 8}, {&h->d_done_stage, n},
                                     {&h->d_info_stage, n * FP_INFO_STRIDE * 8}}));
        const size_t abpe = na * 4 * (act_dtype == FP_F64 ? 8 : 4);          // action bytes per env
        CUDA_TRY(h, cudaMemcpyAsync(h->d_act_stage, h_actions, n * abpe, cudaMemcpyHostToDevice, st));
        int rc = fp_step(h, h->d_act_stage, act_dtype, h->d_reward_stage, h->d_done_stage,
                         h_info ? h->d_info_stage : nullptr, nullptr, stream);
        if (rc != FP_OK) return rc;
        CUDA_TRY(h, cudaMemcpyAsync(h_reward, h->d_reward_stage, n * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(h, cudaMemcpyAsync(h_done, h->d_done_stage, n, cudaMemcpyDeviceToHost, st));
        if (h_info) CUDA_TRY(h, cudaMemcpyAsync(h_info, h->d_info_stage, n * FP_INFO_STRIDE * 8, cudaMemcpyDeviceToHost, st));
    }
    CUDA_TRY(h, cudaStreamSynchronize(st));
    return FP_OK;
}

static void fill_obs_params(FpHandle* h, ObsParams& p, void* out, int push) {
    std::memset(&p, 0, sizeof(p));
    p.c = h->dc; p.n = h->n; p.P = h->d_P; p.Q = h->d_Q; p.PVP = h->d_PVP; p.OBSROW = h->d_OBS;
    p.rec = h->d_rec; p.V = h->d_V; p.hist = h->d_hist;
    for (int i = 0; i < 8; ++i) p.agent_col[i] = h->topo.agent_col[i];
    p.out = out; p.push = push;
}

// The fp64 history ring after ring-only steps (fp_set_obs_history(h, 0)): restored from the env-minor ring, which is
// valid whenever the history is not.
static int hist_ensure(FpHandle* h, cudaStream_t st) {
    if (h->hist_valid) return FP_OK;
    if (!h->d_obsr || !h->obsr_valid) return fail(h, FP_ESTATE, "observation history lost: neither the fp64 ring nor the env-minor ring is valid");
    ObsParams p; fill_obs_params(h, p, nullptr, 0);
    CUDA_TRY(h, launch_hist_from_ring(p, h->d_obsr, h->n_pad, h->ring_q, st));
    h->launches++;
    h->hist_valid = true;
    return FP_OK;
}

int fp_set_obs_history(FpHandle* h, int keep) {
    if (!h) return FP_EINVAL;
    h->keep_hist = keep ? 1 : 0;
    return FP_OK;
}

int fp_get_obs(FpHandle* h, void* d_out, int dtype, int push, void* stream) {
    ENV_ENTRY(h, "fp_get_obs");
    if (!d_out || (dtype != FP_F32 && dtype != FP_F64)) return fail(h, FP_EINVAL, "fp_get_obs: bad arguments");
    { const int rc = hist_ensure(h, (cudaStream_t)stream); if (rc != FP_OK) return rc; }
    ObsParams p; fill_obs_params(h, p, d_out, push ? 1 : 0);
    CUDA_TRY(h, launch_obs(p, dtype == FP_F64, h->grid_obs, (cudaStream_t)stream));
    h->launches++;
    if (push) { h->obsm_valid = false; h->obsr_valid = false; }   // the fp32 rings missed this push: rebuilt on their next use
    return FP_OK;
}

// Window ring bookkeeping: make the ring usable (allocate / rebuild) and, for a push, advance the write
// slot (compacting at the end of the ring).  Returns the slot the push writes.
static int obs_ring_prepare(FpHandle* h, bool push, cudaStream_t st) {
    const int H = h->dc.history, na = h->dc.na;
    const int64_t per_env = (int64_t)na * 3 * H * 6;
    { const int rc = hist_ensure(h, st); if (rc != FP_OK) return rc; }   // the rebuild and the push below use the fp64 ring
    ObsParams p; fill_obs_params(h, p, nullptr, 1);
    if (!h->d_obsm) {
        CUDA_TRY(h, cudaMalloc(&h->d_obsm, (size_t)h->n * per_env * 4));
        h->obsm_valid = false;
    }
    if (!h->obsm_valid) {                          // (re)build from the fp64 history ring: state after a push at w = H - 1
        CUDA_TRY(h, launch_obsm_rebuild(p, h->d_obsm, st));
        h->launches++;
        h->obs_q = H - 1; h->obsm_valid = true;
    }
    if (push) {
        if (h->obs_q == 3 * H - 1) {               // end of the ring: the last H-1 entries move to the front
            CUDA_TRY(h, launch_obsm_compact(h->d_obsm, h->n * na, H, st));
            h->launches++;
            h->obs_q = H - 2;
        }
        h->obs_q += 1;
    }
    return FP_OK;
}

int fp_get_obs_view(FpHandle* h, int push, float** d_view, int64_t* env_pitch, int64_t* agent_pitch, void* stream) {
    if (!d_view) return FP_EINVAL;
    ENV_ENTRY(h, "fp_get_obs_view");
    const int H = h->dc.history, na = h->dc.na;
    cudaStream_t st = (cudaStream_t)stream;
    int rc = obs_ring_prepare(h, push != 0, st);
    if (rc != FP_OK) return rc;
    if (push) {
        ObsParams p; fill_obs_params(h, p, nullptr, 1);
        CUDA_TRY(h, launch_obs_push(p, h->d_obsm, h->obs_q, h->grid_obs, st));
        h->launches++;
        h->obsr_valid = false;
    }
    *d_view = h->d_obsm + (int64_t)(h->obs_q - H + 1) * 6;    // slots w-H+1 .. w: oldest .. newest
    if (env_pitch) *env_pitch = (int64_t)na * 3 * H * 6;
    if (agent_pitch) *agent_pitch = (int64_t)3 * H * 6;
    return FP_OK;
}

/* step + the pushing get_obs that follows it in the rollout loop, dense-view form: two launches (the one-launch
 * form pushes into the env-minor ring, fp_step_ring) */
int fp_step_obs(FpHandle* h, const void* d_actions, int act_dtype, double* d_reward, uint8_t* d_done, double* d_info,
                const uint8_t* d_mask, float** d_view, int64_t* env_pitch, int64_t* agent_pitch, void* stream) {
    if (!h || !d_view) return FP_EINVAL;
    int rc = fp_step(h, d_actions, act_dtype, d_reward, d_done, d_info, d_mask, stream);
    if (rc != FP_OK) return rc;
    return fp_get_obs_view(h, 1, d_view, env_pitch, agent_pitch, stream);
}

// Env-minor ring bookkeeping: allocate / rebuild from the fp64 history ring; for a push, advance the slot.
static int obs_envminor_prepare(FpHandle* h, bool push, cudaStream_t st) {
    const int H = h->dc.history, na = h->dc.na;
    if (!h->d_obsr) {
        h->n_pad = (h->n + 31) / 32 * 32;
        CUDA_TRY(h, cudaMalloc(&h->d_obsr, (size_t)H * na * 6 * h->n_pad * 4));
        h->obsr_valid = false;
    }
    if (!h->obsr_valid) {
        if (!h->hist_valid) return fail(h, FP_ESTATE, "observation history lost: neither the fp64 ring nor the env-minor ring is valid");
        ObsParams p; fill_obs_params(h, p, nullptr, 1);
        CUDA_TRY(h, launch_obsr_rebuild(p, h->d_obsr, h->n_pad, st));
        h->launches++;
        h->ring_q = H - 1; h->obsr_valid = true;
    }
    if (push) h->ring_q = (h->ring_q + 1) % H;
    return FP_OK;
}

int fp_obs_ring(FpHandle* h, float** d_ring, int32_t* slot, int64_t* n_pad, void* stream) {
    if (!d_ring) return FP_EINVAL;
    ENV_ENTRY(h, "fp_obs_ring");
    int rc = obs_envminor_prepare(h, false, (cudaStream_t)stream);
    if (rc != FP_OK) return rc;
    *d_ring = h->d_obsr;
    if (slot) *slot = h->ring_q;
    if (n_pad) *n_pad = h->n_pad;
    return FP_OK;
}

int fp_step_ring(FpHandle* h, const void* d_actions, int act_dtype, double* d_reward, uint8_t* d_done, double* d_info,
                 const uint8_t* d_mask, float** d_ring, int32_t* slot, int64_t* n_pad, void* stream) {
    if (!d_ring) return FP_EINVAL;
    ENV_ENTRY(h, "fp_step_ring");
    // one launch for the built-in feeder shape; the run-time-table kernels, the warp variant and masked steps push
    // through the generic path (fp64 history ring) and rebuild the ring from it: same contents
    const bool fuse = (h->variant == FP_VARIANT_THREAD) && d_mask == nullptr && h->shape == SHAPE_IEEE33;
    if (!fuse) {
        int rc = fp_step(h, d_actions, act_dtype, d_reward, d_done, d_info, d_mask, stream);
        if (rc != FP_OK) return rc;
        float* view = nullptr;
        rc = fp_get_obs_view(h, 1, &view, nullptr, nullptr, stream);
        if (rc != FP_OK) return rc;
        return fp_obs_ring(h, d_ring, slot, n_pad, stream);
    }
    int rc = obs_envminor_prepare(h, true, (cudaStream_t)stream);
    if (rc != FP_OK) return rc;
    h->fuse_obs = 1;
    rc = fp_step(h, d_actions, act_dtype, d_reward, d_done, d_info, nullptr, stream);
    h->fuse_obs = 0;
    if (rc != FP_OK) return rc;
    if (!h->keep_hist) h->hist_valid = false;      // ring-only stepping: the fp64 history ring missed this push (hist_ensure)
    h->obsm_valid = false;                         // the env-major window ring missed this push
    *d_ring = h->d_obsr;
    if (slot) *slot = h->ring_q;
    if (n_pad) *n_pad = h->n_pad;
    return FP_OK;
}

int fp_obs_ring_reset_push(FpHandle* h, const uint8_t* d_mask, void* stream) {
    ENV_ENTRY(h, "fp_obs_ring_reset_push");
    int rc = obs_envminor_prepare(h, false, (cudaStream_t)stream);
    if (rc != FP_OK) return rc;
    ObsParams p; fill_obs_params(h, p, nullptr, 1);
    CUDA_TRY(h, launch_obsr_reset_push(p, h->d_obsr, h->n_pad, h->ring_q, d_mask, (cudaStream_t)stream));
    h->launches++;
    h->obsm_valid = false;
    return FP_OK;
}

int fp_obs_ring_gather(FpHandle* h, float* d_out, void* stream) {
    if (!d_out) return FP_EINVAL;
    ENV_ENTRY(h, "fp_obs_ring_gather");
    int rc = obs_envminor_prepare(h, false, (cudaStream_t)stream);
    if (rc != FP_OK) return rc;
    CUDA_TRY(h, launch_obsr_gather(h->d_obsr, d_out, h->n, h->n_pad, h->dc.na, h->dc.history, h->ring_q, (cudaStream_t)stream));
    h->launches++;
    return FP_OK;
}

// Safety layer (madrl/models/safemaddpg.py:176-299) as a batched closed-form projection: see k_safety_project.
int fp_safety_load(FpHandle* h, const double* h_coef, const double* h_intercept, double v_min, double v_max, double slack_weight) {
    if (!h) return FP_EINVAL;
    if (!h_coef || !h_intercept) return fail(h, FP_EINVAL, "fp_safety_load: null model");
    if (!(slack_weight > 0.0) || !(v_min < v_max)) return fail(h, FP_EINVAL, "fp_safety_load: bad limits / weight");
    const int nb = h->dc.nb, na = h->dc.na;
    // safemaddpg.py:182-184: W_P = coef[:, :nb], W_Q = coef[:, nb:]; :266,272 multiply their ROW SUMS by the bus's own P_net / Q_net
    for (int i = 0; i < na; ++i) {
        const int bus = h->topo.agent_col[i] + 1;                 // bus position of agent i's building
        double sp = 0.0, sq = 0.0;
        for (int j = 0; j < nb; ++j) { sp += h_coef[(size_t)bus * 2 * nb + j]; sq += h_coef[(size_t)bus * 2 * nb + nb + j]; }
        h->safety_sP[i] = sp; h->safety_sQ[i] = sq; h->safety_b[i] = h_intercept[bus];
    }
    h->safety_vmin = v_min; h->safety_vmax = v_max; h->safety_w = slack_weight; h->safety_loaded = 1;
    return FP_OK;
}

int fp_safety_project(FpHandle* h, const void* d_actions, int act_dtype, float* d_adjusted, int32_t type_major, double* d_slack,
                      uint8_t* d_intervened, void* stream) {
    if (h && !h->safety_loaded) return fail(h, FP_ESTATE, "fp_safety_project: call fp_safety_load first");
    ENV_ENTRY(h, "fp_safety_project");
    if (!d_actions || !d_adjusted || (act_dtype != FP_F32 && act_dtype != FP_F64)) return fail(h, FP_EINVAL, "fp_safety_project: bad arguments");
    SafetyParams p;
    std::memset(&p, 0, sizeof(p));
    fill_obs_params(h, p.o, nullptr, 0);
    for (int i = 0; i < h->dc.na; ++i) { p.sP[i] = h->safety_sP[i]; p.sQ[i] = h->safety_sQ[i]; p.b[i] = h->safety_b[i]; }
    p.v_min = h->safety_vmin; p.v_max = h->safety_vmax; p.w = h->safety_w;
    p.actions = d_actions; p.act_f64 = (act_dtype == FP_F64);
    p.out = d_adjusted; p.type_major = type_major; p.slack = d_slack; p.intervened = d_intervened;
    CUDA_TRY(h, launch_safety_project(p, (cudaStream_t)stream));
    h->launches++;
    return FP_OK;
}

// The safety layer against the full affine map V = A [P_1, Q_1, ..., P_nb, Q_nb] + c: see k_safety_project_affine.
int fp_safety_load_affine(FpHandle* h, int32_t n_in, int32_t n_out, const double* h_A, const double* h_c, double v_min,
                          double v_max, double slack_weight) {
    if (!h) return FP_EINVAL;
    USE_DEVICE(h);
    const int nb = h->dc.nb;
    if (!h_A || !h_c) return fail(h, FP_EINVAL, "fp_safety_load_affine: null map");
    if (n_in != 2 * nb || n_out != nb) return fail(h, FP_EINVAL, "fp_safety_load_affine: the map must be [n_bus][2 n_bus]");
    if (!(slack_weight > 0.0) || !std::isfinite(slack_weight) || !(v_min < v_max) || !std::isfinite(v_min) || !std::isfinite(v_max))
        return fail(h, FP_EINVAL, "fp_safety_load_affine: bad limits / weight");
    std::vector<double> At((size_t)2 * nb * FP_MAX_BUS, 0.0);
    for (int n = 0; n < nb; ++n) {
        if (!std::isfinite(h_c[n])) return fail(h, FP_EINVAL, "fp_safety_load_affine: non-finite intercept");
        for (int j = 0; j < 2 * nb; ++j) {
            const double v = h_A[(size_t)n * 2 * nb + j];
            if (!std::isfinite(v)) return fail(h, FP_EINVAL, "fp_safety_load_affine: non-finite map entry");
            At[(size_t)j * FP_MAX_BUS + n] = v;
        }
    }
    h->saff_loaded = 0;
    if (!h->d_saff_At)
        CUDA_TRY(h, alloc_group({{&h->d_saff_At, (size_t)2 * FP_MAX_BUS * FP_MAX_BUS * sizeof(double)},
                                 {&h->d_saff_c, FP_MAX_BUS * sizeof(double)}}));
    CUDA_TRY(h, cudaMemcpy(h->d_saff_At, At.data(), At.size() * sizeof(double), cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->d_saff_c, h_c, (size_t)nb * sizeof(double), cudaMemcpyHostToDevice));
    h->saff_vmin = v_min; h->saff_vmax = v_max; h->saff_w = slack_weight; h->saff_loaded = 1;
    return FP_OK;
}

int fp_safety_project_affine(FpHandle* h, const void* d_actions, int act_dtype, float* d_adjusted, int32_t type_major,
                             double* d_slack, uint8_t* d_intervened, int32_t* d_status, void* stream) {
    if (h && !h->saff_loaded) return fail(h, FP_ESTATE, "fp_safety_project_affine: call fp_safety_load_affine first");
    ENV_ENTRY(h, "fp_safety_project_affine");
    if (!d_actions || !d_adjusted || (act_dtype != FP_F32 && act_dtype != FP_F64))
        return fail(h, FP_EINVAL, "fp_safety_project_affine: bad arguments");
    SafetyAffineParams p;
    std::memset(&p, 0, sizeof(p));
    fill_obs_params(h, p.o, nullptr, 0);
    p.At = h->d_saff_At; p.cvec = h->d_saff_c;
    p.v_min = h->saff_vmin; p.v_max = h->saff_vmax; p.w = h->saff_w;
    p.actions = d_actions; p.act_f64 = (act_dtype == FP_F64);
    p.out = d_adjusted; p.type_major = type_major; p.slack = d_slack; p.intervened = d_intervened; p.status = d_status;
    CUDA_TRY(h, launch_safety_project_affine(p, (cudaStream_t)stream));
    h->launches++;
    return FP_OK;
}

int fp_get_state(FpHandle* h, void* d_out, int dtype, void* stream) {
    ENV_ENTRY(h, "fp_get_state");
    if (!d_out || (dtype != FP_F32 && dtype != FP_F64)) return fail(h, FP_EINVAL, "fp_get_state: bad arguments");
    ObsParams p; fill_obs_params(h, p, d_out, 0);
    CUDA_TRY(h, launch_state(p, dtype == FP_F64, h->grid_obs, (cudaStream_t)stream));
    h->launches++;
    return FP_OK;
}

int fp_state_ptrs(FpHandle* h, void** d_rec, void** d_voltage, void** d_setpoint, void** d_pflow,
                  void** d_qflow, void** d_isq) {
    if (!h) return FP_EINVAL;
    if (d_rec) *d_rec = h->d_rec;
    if (d_voltage) *d_voltage = h->d_V;
    if (d_setpoint) *d_setpoint = h->d_setp;
    if (d_pflow) *d_pflow = h->d_pfl;
    if (d_qflow) *d_qflow = h->d_qfl;
    if (d_isq) *d_isq = h->d_isq;
    return FP_OK;
}

// The fp64 observation-history ring (the source of truth of get_obs, quirk Q7): [N][history][FP_HIST_SLOT] doubles.
// With write != 0 the caller is about to overwrite it (state restore): the derived fp32 rings are rebuilt on next use.
int fp_history_ptr(FpHandle* h, void** d_hist, int64_t* doubles_per_env, int32_t write) {
    if (!h || !d_hist) return FP_EINVAL;
    USE_DEVICE(h);
    if (write) h->hist_valid = true;               // about to be overwritten as a whole
    else { const int rc = hist_ensure(h, nullptr); if (rc != FP_OK) return rc; CUDA_TRY(h, cudaStreamSynchronize(nullptr)); }
    *d_hist = h->d_hist;
    if (doubles_per_env) *doubles_per_env = (int64_t)h->dc.history * FP_HIST_SLOT;
    if (write) { h->obsm_valid = false; h->obsr_valid = false; }
    return FP_OK;
}

int fp_set_keep_flows(FpHandle* h, int keep) {
    if (!h) return FP_EINVAL;
    if (keep && !h->d_pfl) {
        USE_DEVICE(h);
        const size_t bytes = (size_t)h->n * h->dc.nl * 8;
        CUDA_TRY(h, alloc_group({{&h->d_pfl, bytes}, {&h->d_qfl, bytes}, {&h->d_isq, bytes}}, true));
    }
    h->keep_flows = keep ? 1 : 0;
    return FP_OK;
}

int fp_power_flow(FpHandle* h, int64_t n, const double* d_p, const double* d_q, double* d_V, double* d_Pl,
                  double* d_Ql, double* d_Isq, int32_t* d_iters, uint8_t* d_fail, void* stream) {
    if (!h) return FP_EINVAL;
    USE_DEVICE(h);
    if (n < 1 || !d_p || !d_q || !d_V) return fail(h, FP_EINVAL, "fp_power_flow: bad arguments");
    PfParams p;
    p.topo = h->d_topo; p.n = n; p.nl = h->dc.nl; p.max_iter = h->dc.pf_max_iter; p.tol = h->dc.pf_tol; p.n32 = h->dc.pf_f32; p.pad_ = 0;
    p.p = d_p; p.q = d_q; p.V = d_V; p.Pl = d_Pl; p.Ql = d_Ql; p.Isq = d_Isq; p.iters = d_iters; p.fail = d_fail;
    const int cap = h->cap[MODE_PF];
    if (h->variant == FP_VARIANT_THREAD) {                           // grids as launch_env_any's
        PfParamsT pt;
        pt.p = p; pt.t = h->tt;
        const int64_t tiles = (n + 31) / 32;
        CUDA_TRY(h, launch_power_flow_t(h->shape, pt, (int)((tiles < cap) ? tiles : cap), (cudaStream_t)stream));
    } else {
        const int64_t ctas = (n + ENVS_PER_CTA - 1) / ENVS_PER_CTA;
        CUDA_TRY(h, launch_power_flow(p, (int)((ctas < cap) ? ctas : cap), (cudaStream_t)stream));
    }
    h->launches++;
    return FP_OK;
}

int fp_stats_read(FpHandle* h, double* d_out, void* stream) {
    if (!h || !d_out) return FP_EINVAL;
    USE_DEVICE(h);
    CUDA_TRY(h, launch_stats_fold(h->d_stats_partial, h->stats_rows, d_out, (cudaStream_t)stream));
    h->launches++;
    return FP_OK;
}

int fp_stats_reset(FpHandle* h, void* stream) {
    if (!h) return FP_EINVAL;
    USE_DEVICE(h);
    CUDA_TRY(h, cudaMemsetAsync(h->d_stats_partial, 0, (size_t)h->stats_rows * FP_NSTATS * 8, (cudaStream_t)stream));
    return FP_OK;
}

int fp_inject_failure(FpHandle* h, const uint8_t* d_mask) {
    if (!h) return FP_EINVAL;
    h->d_inject = d_mask;
    return FP_OK;
}

}  // extern "C"
