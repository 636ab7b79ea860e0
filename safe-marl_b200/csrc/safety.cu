// safety.cu -- the SAFEMADDPG safety layer against the full affine voltage map (fp_safety_project_affine).
//
// k_safety_project (flex_kernels.cu) projects against the reference's row-sum reading of the regressor, under which
// the QP separates per building.  This kernel solves the problem with the map as it was trained,
// V = A [P_1, Q_1, ..., P_nb, Q_nb] + c, where every bus depends on every building:
//     min_y  sum_k ||y_k - y0_k||^2 + w sum_n [max(0, v_min - V_n(y)) + max(0, V_n(y) - v_max)],  x, c, d >= 0.
// V depends on y only through z = (u_1..u_na, g_1..g_na), u_k = -Pd x_k + c_k - d_k: V = V(y0) + B (z - z0) with
// B[n][k] = A[n][2 b_k], B[n][na + k] = A[n][2 b_k + 1].  For a given u_k the best (x, c, d) is y(r) = max(y0 + (r / 2)
// a, 0), a = (-Pd, 1, -1), the projection k_safety_project uses, so phi_k(u) = min ||y - y0||^2 is C^1 and piecewise
// quadratic in u (phi' = r, phi'' = 1 / s with s = du/dr, <= 3 breakpoints in r).  What is left is a 2 na-variable
// problem, solved by a primal active-set method (mirrored step for step by oracle/safety_affine_ref.py project_affine):
//   * each bus is inside, below (cost -w V), above (+w V) or held at a limit (the working set W, multiplier lam);
//   * one iteration takes the Newton step of the current piece model with V_W held at its limits (|W| x |W| SPD
//     solve, |W| <= 2 na) and walks along it up to the Newton point through the kinks (a bus reaching a limit raises
//     the directional derivative by w |dV_n|) and the buildings' breakpoints (curvature changes); where the derivative
//     turns non-negative on a kink, that bus joins W;
//   * after a full Newton step with nothing crossed, a multiplier outside [0, w] (at v_min) or [-w, 0] (at v_max)
//     releases its bus; none: optimal.  The objective is strictly convex in y, so the optimum is unique.
// Mapping: one warp per env.  Lane l owns buses l and l + 32 (their rows of A), lane k < na owns building k's u_k and
// its piece, lane na + k owns g_k.  A sits transposed in shared memory (17 KB fp64); the small dense algebra runs in
// per-warp shared scratch.  fp64 throughout, no atomics, fixed reduction orders: deterministic.
#include "flex_kernels.cuh"
#include "flex_env_math.cuh"

namespace {

constexpr int SA_WARPS = 8;
constexpr int SA_MAXV = 2 * FP_MAX_AGENTS;             // variables of the reduced problem
constexpr int SA_MAX_ITER = 64;                         // oracle/safety_affine_ref.py AFFINE_MAX_ITER
constexpr double SA_DV_TOL = 1e-12;                     // AFFINE_DV_TOL
constexpr double SA_LAM_TOL = 1e-9;                     // AFFINE_LAM_TOL (relative to w)
enum { ST_IN = 0, ST_LO = 1, ST_HI = 2, ST_AT_MIN = 3, ST_AT_MAX = 4 };

struct SaWarp {
    double x[2 * FP_MAX_BUS];                           // the env's P/Q row at the proposal, interleaved
    double hinv[SA_MAXV], grad[SA_MAXV], p[SA_MAXV], lam[SA_MAXV];
    double V[FP_MAX_BUS];
    double M[SA_MAXV][SA_MAXV + 1];                     // W's system, augmented with its right-hand side
    double w_side[SA_MAXV];                             // +1: held at v_max, -1: at v_min
    int w_bus[SA_MAXV];
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

// (alpha, code) minimum over the warp: smallest alpha, then smallest code (buses 0.., buildings 64..)
__device__ __forceinline__ void warp_argmin(double& a, int& code) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double oa = __shfl_xor_sync(FULL, a, o);
        const int oc = __shfl_xor_sync(FULL, code, o);
        if (oa < a || (oa == a && oc < code)) { a = oa; code = oc; }
    }
}

// piece [lo, hi] of r with index j over the sorted breakpoints b0 <= b1 <= b2
__device__ __forceinline__ void piece_bounds(double b0, double b1, double b2, int j, double& lo, double& hi) {
    const double inf = __longlong_as_double(0x7ff0000000000000ll);
    lo = (j == 0) ? -inf : (j == 1) ? b0 : (j == 2) ? b1 : b2;
    hi = (j == 0) ? b0 : (j == 1) ? b1 : (j == 2) ? b2 : inf;
}

// du/dr on [lo, hi]: a variable with a_i > 0 is free above its breakpoint t_i, one with a_i < 0 below it
__device__ __forceinline__ double piece_slope(const double (&a)[3], const double (&t)[3], double lo, double hi) {
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 3; ++i)
        if ((a[i] > 0.0 && lo >= t[i]) || (a[i] < 0.0 && hi <= t[i])) s += a[i] * a[i] * 0.5;
    return s;
}

__global__ void __launch_bounds__(SA_WARPS * 32) k_safety_project_affine(const SafetyAffineParams prm) {
    __shared__ double s_At[2 * FP_MAX_BUS * FP_MAX_BUS];
    __shared__ SaWarp s_w[SA_WARPS];
    const DevCfg& c = prm.o.c;
    const int nb = c.nb, nl = c.nl, na = c.na, nv = 2 * na;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < 2 * nb * FP_MAX_BUS; i += blockDim.x) s_At[i] = __ldg(prm.At + i);
    __syncthreads();
    SaWarp& sw = s_w[warp];
    const double v_min = prm.v_min, v_max = prm.v_max, w = prm.w;
    const double inf = __longlong_as_double(0x7ff0000000000000ll);
    // the rows of B this lane reads: column of variable i is At[(2 b_k + (i >= na)) * FP_MAX_BUS + n]
    auto Bcol = [&](int i) -> const double* {
        const int k = (i < na) ? i : i - na;
        return s_At + (2 * (prm.o.agent_col[k] + 1) + ((i < na) ? 0 : 1)) * FP_MAX_BUS;
    };
    const bool own1 = lane + 32 < nb;                   // the lane also owns bus lane + 32
    const bool is_u = lane < na, is_g = lane >= na && lane < nv;
    const int ak = is_u ? lane : (is_g ? lane - na : 0);     // building of this lane's variable

    for (int64_t e = (int64_t)blockIdx.x * SA_WARPS + warp; e < prm.o.n; e += (int64_t)gridDim.x * SA_WARPS) {
        // ---- the proposal: the env's current demands and parse_actions (the same calls as k_safety_project)
        const uint64_t* rec = prm.o.rec + e * FP_REC_STRIDE;
        const int64_t row = row_in_force(c, rec);
        double y0[4] = {0.0, 0.0, 0.0, 0.0}, Pd = 0.0;
        if (lane < na) {
            const double* orow = prm.o.OBSROW + row * FP_OBS_STRIDE;
            Pd = __ldg(orow + FP_OBS_P + lane);
            const double ppv = __ldg(orow + FP_OBS_PV + lane);
            const double e_cur = __longlong_as_double((long long)rec[FP_REC_E_CUR + lane]);
            double a0, a1, a2, a3;
            load_action4(prm.actions, prm.act_f64, e * na + lane, a0, a1, a2, a3);
            const Setpoint sp = apply_actions_frac<true>(c, true, a0, a1, a2, a3, ppv, e_cur);
            y0[0] = sp.pred; y0[1] = sp.ch; y0[2] = sp.dis; y0[3] = sp.qpv;
        }
        // full bus-order P/Q row (0 at the slack bus), with the proposal applied at the buildings' buses
        for (int m = lane; m < nb; m += 32) {
            sw.x[2 * m] = (m == 0) ? 0.0 : __ldg(prm.o.P + row * nl + m - 1);
            sw.x[2 * m + 1] = (m == 0) ? 0.0 : __ldg(prm.o.Q + row * nl + m - 1);
        }
        __syncwarp();
        if (lane < na) {
            const int m = prm.o.agent_col[lane] + 1;
            sw.x[2 * m] = Pd * (1.0 - y0[0]) + y0[1] - y0[2];
            sw.x[2 * m + 1] = sw.x[2 * m + 1] + y0[3];
        }
        __syncwarp();
        // ---- V(y0): lane-parallel GEMV over the full row
        double V0[2] = {0.0, 0.0};
#pragma unroll
        for (int sl = 0; sl < 2; ++sl) {
            const int n = lane + 32 * sl;
            if (n < nb) {                                   // four independent chains (2 nb is even), fixed order
                double acc[4] = {0.0, 0.0, 0.0, 0.0};
                for (int j = 0; j < 2 * nb; j += 4) {
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        if (j + q < 2 * nb) acc[q] = fma(s_At[(j + q) * FP_MAX_BUS + n], sw.x[j + q], acc[q]);
                }
                V0[sl] = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + __ldg(prm.cvec + n);
            }
        }
        const bool out0 = V0[0] < v_min || V0[0] > v_max;
        const bool out1 = own1 && (V0[1] < v_min || V0[1] > v_max);
        // a NaN proposal (numpy.clip keeps a NaN action) makes V(y0) non-finite: the env is left as parsed, unprojected
        const bool bad = (lane < nb && !isfinite(V0[0])) || (own1 && !isfinite(V0[1]));
        const bool any_out = __any_sync(FULL, (lane < nb && out0) || out1) && !__any_sync(FULL, bad);
        double y[4] = {y0[0], y0[1], y0[2], y0[3]};
        int status = 0;
        int st[2] = {ST_IN, ST_IN};
        double V[2] = {V0[0], V0[1]};
        if (any_out) {
#pragma unroll
            for (int sl = 0; sl < 2; ++sl) st[sl] = (V0[sl] < v_min) ? ST_LO : ((V0[sl] > v_max) ? ST_HI : ST_IN);
            // building lanes: the piece structure of phi_k
            double a[3] = {-Pd, 1.0, -1.0}, t[3], b0, b1, b2;
#pragma unroll
            for (int i = 0; i < 3; ++i) t[i] = (a[i] != 0.0) ? (-2.0 * y0[i] / a[i]) : inf;
            b0 = t[0]; b1 = t[1]; b2 = t[2];                // sorted by a three-element network
            if (b0 > b1) { const double s_ = b0; b0 = b1; b1 = s_; }
            if (b1 > b2) { const double s_ = b1; b1 = b2; b2 = s_; }
            if (b0 > b1) { const double s_ = b0; b0 = b1; b1 = s_; }
            int piece = (b0 <= 0.0) + (b1 <= 0.0) + (b2 <= 0.0);
            double r = 0.0, dz = 0.0, s = 0.5;
            int m = 0, released = -1;
            double released_lim = 0.0;
            status = -1;
            for (int it = 0; it < SA_MAX_ITER; ++it) {
                double lo, hi;
                if (is_u) { piece_bounds(b0, b1, b2, piece, lo, hi); s = piece_slope(a, t, lo, hi); }
                const double hinv = is_u ? s : 0.5;
                // V at the iterate and the gradient of the current piece model
#pragma unroll
                for (int sl = 0; sl < 2; ++sl) V[sl] = V0[sl];
                for (int i = 0; i < nv; ++i) {
                    const double dzi = __shfl_sync(FULL, dz, i);
                    const double* col = Bcol(i);
                    V[0] = fma(col[lane], dzi, V[0]);
                    if (own1) V[1] = fma(col[lane + 32], dzi, V[1]);
                }
                const double cf0 = (lane < nb) ? ((st[0] == ST_LO) ? w : ((st[0] == ST_HI) ? -w : 0.0)) : 0.0;
                const double cf1 = own1 ? ((st[1] == ST_LO) ? w : ((st[1] == ST_HI) ? -w : 0.0)) : 0.0;
                double grad = 0.0;
                for (int i = 0; i < nv; ++i) {
                    const double* col = Bcol(i);
                    double part = (lane < nb) ? cf0 * col[lane] : 0.0;
                    if (own1) part = fma(cf1, col[lane + 32], part);
                    const double tot = warp_sum(part);
                    if (lane == i) grad = (is_u ? r : 2.0 * dz) - tot;
                }
                if (lane < nv) { sw.hinv[lane] = hinv; sw.grad[lane] = grad; }
                if (lane < nb) sw.V[lane] = V[0];
                if (own1) sw.V[lane + 32] = V[1];
                __syncwarp();
                // Newton step with V_W held at its limits: (B_W H^-1 B_W^T) lam = (t_W - V_W) + B_W H^-1 grad
                if (m > 0) {
                    for (int q = lane; q < m * (m + 1); q += 32) {
                        const int ra = q / (m + 1), cb = q - ra * (m + 1);
                        const int na_ = sw.w_bus[ra];
                        double acc = 0.0;
                        if (cb < m) {
                            const int nb_ = sw.w_bus[cb];
                            for (int i = 0; i < nv; ++i) { const double* col = Bcol(i); acc = fma(col[na_] * sw.hinv[i], col[nb_], acc); }
                        } else {
                            for (int i = 0; i < nv; ++i) { const double* col = Bcol(i); acc = fma(col[na_] * sw.hinv[i], sw.grad[i], acc); }
                            const double tgt = (sw.w_side[ra] > 0.0) ? v_max : v_min;
                            acc += tgt - sw.V[na_];
                        }
                        sw.M[ra][cb] = acc;
                    }
                    __syncwarp();
                    // Gaussian elimination without pivoting (SPD), lane r < m owns row r
                    for (int k = 0; k < m; ++k) {
                        if (lane > k && lane < m) {
                            const double f = sw.M[lane][k] / sw.M[k][k];
                            for (int cb = k + 1; cb < m; ++cb) sw.M[lane][cb] = fma(-f, sw.M[k][cb], sw.M[lane][cb]);
                            sw.M[lane][m] = fma(-f, sw.M[k][m], sw.M[lane][m]);
                        }
                        __syncwarp();
                    }
                    if (lane == 0) {
                        for (int k = m - 1; k >= 0; --k) {
                            double acc = sw.M[k][m];
                            for (int cb = k + 1; cb < m; ++cb) acc = fma(-sw.M[k][cb], sw.lam[cb], acc);
                            sw.lam[k] = acc / sw.M[k][k];
                        }
                    }
                    __syncwarp();
                }
                double p = 0.0;
                if (lane < nv) {
                    const double* col = Bcol(lane);
                    double acc = 0.0;
                    for (int q = 0; q < m; ++q) acc = fma(col[sw.w_bus[q]], sw.lam[q], acc);
                    p = hinv * (acc - grad);
                    sw.p[lane] = p;
                }
                __syncwarp();
                double dV[2] = {0.0, 0.0};
                for (int i = 0; i < nv; ++i) {
                    const double pi = sw.p[i];
                    const double* col = Bcol(i);
                    if (lane < nb) dV[0] = fma(col[lane], pi, dV[0]);
                    if (own1) dV[1] = fma(col[lane + 32], pi, dV[1]);
                }
                // ---- line search up to the Newton point through the kinks and the breakpoints
                double D = warp_sum((lane < nv) ? grad * p : 0.0);
                double kappa = warp_sum((lane < nv) ? p * p / hinv : 0.0);
                double cur = 0.0;
                bool crossed = false, joined = false;
                while (kappa > 0.0) {
                    double ev_a = inf;
                    int code = 1 << 20;
                    if (m < nv) {
#pragma unroll
                        for (int sl = 0; sl < 2; ++sl) {
                            const int n = lane + 32 * sl;
                            if (n >= nb || st[sl] >= ST_AT_MIN || fabs(dV[sl]) <= SA_DV_TOL) continue;
                            double lim;
                            if (dV[sl] > 0.0 && st[sl] != ST_HI) lim = (st[sl] == ST_IN) ? v_max : v_min;
                            else if (dV[sl] < 0.0 && st[sl] != ST_LO) lim = (st[sl] == ST_IN) ? v_min : v_max;
                            else continue;
                            if (n == released && lim == released_lim) continue;
                            const double an = fmax(cur, (lim - V[sl]) / dV[sl]);
                            if (an < ev_a) { ev_a = an; code = n; }
                        }
                    }
                    if (is_u) {
                        const double dr = p / s;
                        piece_bounds(b0, b1, b2, piece, lo, hi);
                        double ak_ = inf;
                        if (dr > 0.0 && hi < inf) ak_ = cur + fmax(0.0, (hi - r) / dr);
                        else if (dr < 0.0 && lo > -inf) ak_ = cur + fmax(0.0, (lo - r) / dr);
                        if (ak_ < ev_a) { ev_a = ak_; code = 64 + lane; }
                    }
                    warp_argmin(ev_a, code);
                    const double stop = crossed ? fmin(1.0, cur - D / kappa) : 1.0;
                    if (code == (1 << 20) || ev_a >= stop) {
                        if (is_u) r = fma(stop - cur, p / s, r);
                        cur = stop;
                        break;
                    }
                    D = fma(kappa, ev_a - cur, D);
                    if (is_u) r = fma(ev_a - cur, p / s, r);
                    cur = ev_a; crossed = true;
                    if (code < 64) {
                        const int n = code, owner = n & 31, sl = n >> 5;
                        const double dVn = __shfl_sync(FULL, sl ? dV[1] : dV[0], owner);
                        const int stn = __shfl_sync(FULL, sl ? st[1] : st[0], owner);
                        // the limit reached: the one the bus was heading for
                        const double lim = (dVn > 0.0) ? ((stn == ST_IN) ? v_max : v_min) : ((stn == ST_IN) ? v_min : v_max);
                        D += w * fabs(dVn);
                        int nst;
                        if (D >= 0.0) {
                            nst = (lim == v_min) ? ST_AT_MIN : ST_AT_MAX;
                            if (lane == 0) { sw.w_bus[m] = n; sw.w_side[m] = (nst == ST_AT_MAX) ? 1.0 : -1.0; }
                            ++m;
                            joined = true;
                        } else {
                            nst = (stn != ST_IN) ? ST_IN : ((lim == v_max) ? ST_HI : ST_LO);
                        }
                        if (lane == owner) { if (sl) st[1] = nst; else st[0] = nst; }
                        __syncwarp();
                        if (joined) break;
                    } else {
                        const int k = code - 64;
                        double dk = 0.0;
                        if (lane == k) {
                            piece_bounds(b0, b1, b2, piece, lo, hi);
                            r = (p > 0.0) ? hi : lo;
                            piece += (p > 0.0) ? 1 : -1;
                            piece_bounds(b0, b1, b2, piece, lo, hi);
                            const double s_new = piece_slope(a, t, lo, hi);
                            dk = p * p * (1.0 / s_new - 1.0 / s);
                            s = s_new;
                        }
                        kappa += __shfl_sync(FULL, dk, k);
                    }
                }
                if (lane < nv) dz = fma(cur, p, dz);
                if (cur > 0.0) released = -1;
                if (crossed || joined) continue;
                // ---- a full Newton step with nothing crossed: check W's multipliers
                double viol = -inf;
                int vi = 1 << 20;
                if (lane < m) {
                    const double l = sw.lam[lane];
                    viol = (sw.w_side[lane] < 0.0) ? fmax(-l, l - w) : fmax(l, -w - l);
                    vi = lane;
                }
                {   // argmax, first index on ties
                    double nv_ = -viol; int ci = vi;
                    warp_argmin(nv_, ci);
                    viol = -nv_; vi = ci;
                }
                if (m == 0 || viol <= SA_LAM_TOL * w) { status = it + 1; break; }
                const int n = sw.w_bus[vi];
                const bool at_min = sw.w_side[vi] < 0.0;
                const double l = sw.lam[vi];
                __syncwarp();
                if (lane == 0) {
                    for (int q = vi; q + 1 < m; ++q) { sw.w_bus[q] = sw.w_bus[q + 1]; sw.w_side[q] = sw.w_side[q + 1]; }
                }
                __syncwarp();
                --m;
                const int nst = at_min ? ((l < 0.0) ? ST_IN : ST_LO) : ((l > 0.0) ? ST_IN : ST_HI);
                if (lane == (n & 31)) { if (n >> 5) st[1] = nst; else st[0] = nst; }
                released = n; released_lim = at_min ? v_min : v_max;
            }
            // ---- the adjusted setpoints and the prediction at them
            double dzf = 0.0;
            if (is_u) {
#pragma unroll
                for (int i = 0; i < 3; ++i) { const double v = fma(0.5 * r, a[i], y0[i]); y[i] = (v > 0.0) ? v : 0.0; }
                dzf = a[0] * (y[0] - y0[0]) + (y[1] - y0[1]) - (y[2] - y0[2]);
            }
            const double dg = __shfl_sync(FULL, dz, (na + ak) & 31);
            if (is_u) y[3] = y0[3] + dg;
            if (is_g) dzf = dz;
#pragma unroll
            for (int sl = 0; sl < 2; ++sl) V[sl] = V0[sl];
            for (int i = 0; i < nv; ++i) {
                const double di = __shfl_sync(FULL, dzf, i);
                const double* col = Bcol(i);
                if (lane < nb) V[0] = fma(col[lane], di, V[0]);
                if (own1) V[1] = fma(col[lane + 32], di, V[1]);
            }
        }
        // ---- outputs
        if (lane < na) {
            if (prm.type_major) {
#pragma unroll
                for (int k = 0; k < 4; ++k) prm.out[e * 4 * na + k * na + lane] = (float)y[k];
            } else {
                reinterpret_cast<float4*>(prm.out)[e * na + lane] = make_float4((float)y[0], (float)y[1], (float)y[2], (float)y[3]);
            }
            if (prm.intervened != nullptr) {                 // bits, not values: an untouched NaN has not moved
                bool mv = false;
#pragma unroll
                for (int k = 0; k < 4; ++k) mv = mv || (__double_as_longlong(y[k]) != __double_as_longlong(y0[k]));
                prm.intervened[e * na + lane] = mv ? 1 : 0;
            }
        }
        if (prm.slack != nullptr) {
#pragma unroll
            for (int sl = 0; sl < 2; ++sl) {
                const int n = lane + 32 * sl;
                if (n < nb) {
                    const double sv = (st[sl] >= ST_AT_MIN) ? 0.0 : (fmax(0.0, v_min - V[sl]) + fmax(0.0, V[sl] - v_max));
                    prm.slack[e * nb + n] = any_out ? sv : 0.0;
                }
            }
        }
        if (prm.status != nullptr && lane == 0) prm.status[e] = status;
        __syncwarp();
    }
}

}  // namespace

cudaError_t launch_safety_project_affine(const SafetyAffineParams& prm, cudaStream_t st) {
    const int64_t ctas = (prm.o.n + SA_WARPS - 1) / SA_WARPS;
    int per_sm = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_safety_project_affine, SA_WARPS * 32, 0);
    if (e != cudaSuccess) return e;
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int64_t cap = (int64_t)sms * (per_sm > 0 ? per_sm : 1);
    k_safety_project_affine<<<(unsigned)(ctas < cap ? ctas : cap), SA_WARPS * 32, 0, st>>>(prm);
    return cudaGetLastError();
}
