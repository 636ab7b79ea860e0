/*
 * flex_oracle.c -- CPU mirror of the flex_provision hot path.  TEST INFRASTRUCTURE ONLY.
 *
 * PARITY: the reference (kosmylo/Safe-MARL) has no tests or golden vectors for this path and
 * its power flow runs inside IPOPT, which is not available here; the fixtures this mirror is
 * checked against (tests/golden/ref_*.npz) are outputs of the reference's own Python code with
 * only the IPOPT root finder substituted (see oracle/__init__.py).  This file
 * restates the algorithm in plain C, in fp64, with the SAME floating-point operation order
 * as the CUDA kernels (explicit fma(), -ffp-contract=off), so that integer outputs
 * (voltage-violation masks and counts, flags, iteration counts) can be compared bit for
 * bit and floating-point outputs to the last ulp.  Its mathematical correctness is pinned
 * separately by oracle/pf_ref.py (dense Newton on utils/pf.py:65-98) and the literature
 * IEEE-33 known answers (tests/test_oracle_*.py).
 *
 * Reference lines followed:
 *   fo_power_flow   utils/pf.py:115-192 (equations :155-178, outputs :187-190)
 *   fo_env_reset    flexibility_provision_env.py:74-155 (+ :609-619 row load, quirk Q1)
 *   fo_env_step     flexibility_provision_env.py:241-356, reward :679-706,
 *                   ESS update utils/pf.py:96-98
 *   setpoints()     :262-293, :621-626, :628-661, :663-674, :676-677
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference may
 * load this library.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define NL 32
#define ANC_NONE 32u

typedef struct {
    int32_t nb, nl, na, history, episode_limit, raw_actions, pf_max_iter, variant;   /* variant: 0 = thread-per-env order, 1 = warp-per-env order */
    int32_t pf_f32, pad_;        /* thread order: opening passes of a solve that run in fp32 */
    double pf_tol, v_min, v_max, e_min, e_max, p_ch_max, p_dis_max, eta_ch, eta_dis;
    double mpr, kappa, pv_cost, ess_cost, discomfort_coeff, voltage_coeff, delta_t, fail_penalty, e_next_lb;
    /* lane tables (pre-order; lane k <-> bus position col[k]+1) */
    double R[NL], X[NL], Z2[NL], imax2[NL];
    int32_t end[NL], col[NL], agent[NL], anc[5][NL];
    int32_t agent_lane[8], agent_col[8];
    /* thread-per-env tables: lane of the parent line (-1: the slack bus feeds this line) */
    int32_t par[NL];
} FoNet;

/* Build lane tables from bus-order arrays: parent[nb] (-1 for slack at 0), r/x/imax[nb]. */
int fo_build(FoNet* t, int nb, int na, const int32_t* parent, const double* r, const double* x,
             const double* imax, const int32_t* agent_bus) {
    int nl = nb - 1, lane_of[64], bus_of[64], size[64], stack[64], sp = 0, next = 0;
    if (nb < 2 || nb > 33 || parent[0] != -1) return -1;
    for (int b = 0; b < nb; ++b) { lane_of[b] = -1; size[b] = 1; }
    /* pre-order, children in ascending bus position */
    for (int b = nb - 1; b >= 1; --b) if (parent[b] == 0) stack[sp++] = b;
    while (sp > 0) {
        int b = stack[--sp];
        lane_of[b] = next; bus_of[next] = b; ++next;
        for (int k = nb - 1; k >= 1; --k) if (parent[k] == b) stack[sp++] = k;
    }
    if (next != nl) return -2;
    for (int k = nl - 1; k >= 0; --k) { int b = bus_of[k]; if (parent[b] != 0) size[parent[b]] += size[b]; }
    for (int k = 0; k < NL; ++k) {
        t->R[k] = t->X[k] = t->Z2[k] = 0.0; t->imax2[k] = INFINITY;
        t->end[k] = k; t->col[k] = 0; t->agent[k] = -1; t->par[k] = -1;
        for (int j = 0; j < 5; ++j) t->anc[j][k] = ANC_NONE;
    }
    for (int k = 0; k < nl; ++k) {
        int b = bus_of[k];
        t->R[k] = r[b]; t->X[k] = x[b];
        t->par[k] = parent[b] > 0 ? lane_of[parent[b]] : -1;
        t->Z2[k] = r[b] * r[b] + x[b] * x[b];
        t->imax2[k] = imax[b] > 0.0 ? imax[b] * imax[b] : INFINITY;
        t->end[k] = k + size[b] - 1;
        t->col[k] = b - 1;
        for (int j = 0; j < 5; ++j) {
            int a = b;
            for (int s = 0; s < (1 << j) && a > 0; ++s) a = parent[a];
            t->anc[j][k] = a > 0 ? lane_of[a] : (int32_t)ANC_NONE;
        }
    }
    for (int i = 0; i < na; ++i) {
        int b = agent_bus[i];
        if (b < 1 || b >= nb) return -3;
        t->agent[lane_of[b]] = i; t->agent_lane[i] = lane_of[b]; t->agent_col[i] = b - 1;
    }
    t->nb = nb; t->nl = nl; t->na = na;
    return 0;
}

/* Hillis-Steele inclusive scan exactly as 5 rounds of shfl_up + add. */
static void scan32(double* s) {
    for (int d = 1; d < 32; d <<= 1)
        for (int k = 31; k >= d; --k) s[k] = s[k] + s[k - d];
}

typedef struct { double P[NL], Q[NL], ell[NL], v[NL]; int iters; int ok; } Sweep;

/* Lane arrays p, q (length 32, zero beyond nl). */
static void sweep_w(const FoNet* t, const double* p, const double* q, double tol, int max_iter, Sweep* o) {
    double ell[NL], v_old[NL], SP[NL], SQ[NL], d[NL], dn[NL];
    int conv = 0, bad = 0, it = 0;
    for (int k = 0; k < NL; ++k) { ell[k] = 0.0; v_old[k] = 1.0; o->P[k] = o->Q[k] = 0.0; o->v[k] = 1.0; }
    while (it < max_iter) {
        ++it;
        for (int k = 0; k < NL; ++k) { SP[k] = fma(t->R[k], ell[k], p[k]); SQ[k] = fma(t->X[k], ell[k], q[k]); }
        scan32(SP); scan32(SQ);
        for (int k = 0; k < NL; ++k) {
            o->P[k] = p[k] + (SP[t->end[k]] - SP[k]);
            o->Q[k] = q[k] + (SQ[t->end[k]] - SQ[k]);
        }
        for (int k = 0; k < NL; ++k) {
            double x = t->R[k] * o->P[k];
            x = fma(t->X[k], o->Q[k], x);
            d[k] = fma(t->Z2[k], ell[k], x + x);
        }
        for (int r = 0; r < 5; ++r) {                 /* pointer jumping over 2^r-th ancestors */
            for (int k = 0; k < NL; ++k) {
                int a = t->anc[r][k];
                dn[k] = (a < (int)ANC_NONE) ? d[k] + d[a] : d[k];
            }
            memcpy(d, dn, sizeof(d));
        }
        conv = 1; bad = 0;
        for (int k = 0; k < NL; ++k) {
            double v = 1.0 - d[k];
            double s = o->P[k] * o->P[k];
            s = fma(o->Q[k], o->Q[k], s);
            ell[k] = s / v;
            if (!(v > 0.0)) bad = 1;
            if (!(fabs(v - v_old[k]) <= tol)) conv = 0;
            v_old[k] = v; o->v[k] = v;
        }
        if (bad || conv) break;
    }
    memcpy(o->ell, ell, sizeof(ell));
    o->iters = it; o->ok = conv && !bad;
}


/* ---- thread-per-env operation order (variant 0) ------------------------------------------
 * One CUDA thread owns one env and walks the lines in DFS pre-order, ONE pass per iteration.
 * The balance rows (utils/pf.py:65-83) give P_k = S_k + W_k with
 *     S_k = sum of p over the subtree of line k                      (once per solve)
 *     W_k = sum of R_j l_j over the lines strictly below k           (carried down the tree)
 * Lines are grouped in chains (maximal first-child paths; a lateral's first line starts a new
 * chain); U_c is the loss total of the subtree hanging off chain c's first line.
 *   setup   (k = nl-1 .. 0): S_k = (p_k + [S of the non-adjacent children, latest subtree first])
 *                                  + [S_{k+1} if line k+1 is a child of k]
 *   pass    (k = 0 .. nl-1): chain head:  W = U_c,  v_parent = 1 or v of the branch bus
 *                            otherwise:   W = W_{k-1} - U_c' for every chain c' leaving the bus
 *                                         between k-1 and k (increasing c'),  v_parent = v_{k-1}
 *                            W = fma(-R_k, l_k, W);  P = S_k + W   (same for Q with X)
 *                            v_k = fma(-2, fma(Z2/2, l, fma(X, Q, R*P)), v_parent) (pf.py:90-94)
 *                            e = fma(-v_k, l_k, P^2 + Q^2)   residual of the current row (pf.py:85-88)
 *                            l_k' = fma(e, 1 + d + d^2, l_k),  d = 1 - v_k: a division-free
 *                            relaxation whose fixed point is the row itself (1 + d + d^2 =
 *                            (1 - d^3)/v, so it converges like the exact quotient)
 *                            acc_c = fma(R_k, l_k', acc_c)
 *           then, c = n_chains-1 .. 0: U_c = acc_c + U_c' for the chains c' attached to chain c
 *           (increasing c'); stop when max_k |e_k| < tol, compared on the high words of the
 *           fp64 bit patterns (tol to 20 mantissa bits; an integer compare on the GPU)
 *   final   one more pass with the converged l: P, Q, v that satisfy the balance and
 *           voltage-drop rows to rounding (no current update). */
/* v <= 0 (also -0 and the smallest denormals), +-inf or NaN */
static int sqv_bad(double v) {
    uint64_t u;
    memcpy(&u, &v, 8);
    return (uint32_t)((uint32_t)(u >> 32) - 1u) >= 0x7FEFFFFFu;
}

/* high word of |x|'s bit pattern: the convergence measure (NaN maps above every finite value) */
static int32_t hi_abs(double x) {
    uint64_t u;
    memcpy(&u, &x, 8);
    return (int32_t)((u >> 32) & 0x7FFFFFFFu);
}

#define MAXCH 32
typedef struct { int n, chain_of[NL], head[NL]; uint32_t attach[NL], child[MAXCH]; } Chains;

static void chains_of(const FoNet* t, Chains* c) {
    c->n = 0;
    for (int k = 0; k < NL; ++k) { c->chain_of[k] = 0; c->head[k] = 0; c->attach[k] = 0; }
    for (int k = 0; k < MAXCH; ++k) c->child[k] = 0;
    for (int k = 0; k < t->nl; ++k) {
        if (k == 0 || t->par[k] != k - 1) {
            int id = c->n++;
            c->chain_of[k] = id; c->head[k] = 1;
            if (t->par[k] >= 0) { c->attach[t->par[k]] |= 1u << id; c->child[c->chain_of[t->par[k]]] |= 1u << id; }
        } else c->chain_of[k] = c->chain_of[k - 1];
    }
}

static void setup_t(const FoNet* t, const double* p, const double* q, double* SP, double* SQ) {
    double accP[NL], accQ[NL]; int has[NL];
    for (int k = 0; k < NL; ++k) has[k] = 0;
    for (int k = t->nl - 1; k >= 0; --k) {
        double tp = p[k], tq = q[k];
        if (has[k]) { tp = tp + accP[k]; tq = tq + accQ[k]; }
        if (k + 1 < t->nl && t->par[k + 1] == k) { tp = tp + SP[k + 1]; tq = tq + SQ[k + 1]; }
        SP[k] = tp; SQ[k] = tq;
        int a = t->par[k];
        if (a >= 0 && a != k - 1) {                   /* non-adjacent child: deposit into the parent's slot */
            if (has[a]) { accP[a] = accP[a] + tp; accQ[a] = accQ[a] + tq; }
            else { accP[a] = tp; accQ[a] = tq; has[a] = 1; }
        }
    }
}

/* flows and squared voltage of line k; W carried in (wP, wQ) */
static void line_t(const FoNet* t, const Chains* ch, int k, const double* SP, const double* SQ, double ell,
                   const double* UP, const double* UQ, double* wP, double* wQ, double* v, double* P, double* Q) {
    double w, wq, vp;
    if (ch->head[k]) {
        w = UP[ch->chain_of[k]]; wq = UQ[ch->chain_of[k]];
        vp = t->par[k] >= 0 ? v[t->par[k]] : 1.0;
    } else {
        w = *wP; wq = *wQ; vp = v[k - 1];
        for (int c = 0; c < ch->n; ++c) if ((ch->attach[k - 1] >> c) & 1u) { w = w - UP[c]; wq = wq - UQ[c]; }
    }
    w = fma(-t->R[k], ell, w); wq = fma(-t->X[k], ell, wq);
    *wP = w; *wQ = wq;
    *P = SP[k] + w; *Q = SQ[k] + wq;
    double g = t->R[k] * *P;                         /* v_parent - 2 g: scaling by two is exact, so this is */
    g = fma(t->X[k], *Q, g);                         /* fma(Z2, l, fma(2X, Q, 2R*P)) bit for bit            */
    g = fma(0.5 * t->Z2[k], ell, g);
    v[k] = fma(-2.0, g, vp);
}

static void sweep_t(const FoNet* t, const double* p, const double* q, double tol, int max_iter, Sweep* o) {
    double ell[NL], v[NL], SP[NL], SQ[NL], UP[MAXCH], UQ[MAXCH], aP[MAXCH], aQ[MAXCH];
    Chains ch;
    int conv = 0, bad = 0, it = 0;
    chains_of(t, &ch);
    for (int k = 0; k < NL; ++k) { ell[k] = 0.0; v[k] = 1.0; o->P[k] = o->Q[k] = 0.0; SP[k] = SQ[k] = 0.0; }
    for (int c = 0; c < MAXCH; ++c) UP[c] = UQ[c] = 0.0;
    setup_t(t, p, q, SP, SQ);
    if (t->pf_f32 > 0) {
        /* fp32 opening passes (t_open_f32 in flex_thread_kernels.cu): the same pass in IEEE fp32 -- S, the line
         * constants and every intermediate rounded to float, explicit fmaf -- without a convergence test; the
         * currents and the chain loss totals are then widened exactly and the fp64 passes take over */
        float lf[NL], vf[NL], SPf[NL], SQf[NL], UPf[MAXCH], UQf[MAXCH], aPf[MAXCH], aQf[MAXCH];
        for (int k = 0; k < NL; ++k) { lf[k] = 0.0f; vf[k] = 1.0f; SPf[k] = (float)SP[k]; SQf[k] = (float)SQ[k]; }
        for (int c = 0; c < MAXCH; ++c) UPf[c] = UQf[c] = 0.0f;
        for (int n = 0; n < t->pf_f32; ++n) {
            float wP = 0.0f, wQ = 0.0f;
            for (int c = 0; c < MAXCH; ++c) aPf[c] = aQf[c] = 0.0f;
            for (int k = 0; k < t->nl; ++k) {
                const float R = (float)t->R[k], X = (float)t->X[k], Z2h = (float)(0.5 * t->Z2[k]);
                float w, wq, vp;
                if (ch.head[k]) {
                    w = UPf[ch.chain_of[k]]; wq = UQf[ch.chain_of[k]];
                    vp = t->par[k] >= 0 ? vf[t->par[k]] : 1.0f;
                } else {
                    w = wP; wq = wQ; vp = vf[k - 1];
                    for (int c = 0; c < ch.n; ++c) if ((ch.attach[k - 1] >> c) & 1u) { w = w - UPf[c]; wq = wq - UQf[c]; }
                }
                w = fmaf(-R, lf[k], w); wq = fmaf(-X, lf[k], wq);
                wP = w; wQ = wq;
                const float P = SPf[k] + w, Q = SQf[k] + wq;
                float g = R * P;
                g = fmaf(X, Q, g);
                g = fmaf(Z2h, lf[k], g);
                const float vk = fmaf(-2.0f, g, vp);
                vf[k] = vk;
                float sq = P * P;
                sq = fmaf(Q, Q, sq);
                const float e = fmaf(-vk, lf[k], sq);
                const float d = 1.0f - vk;
                float rt = 2.0f - vk;
                rt = fmaf(d, rt, 1.0f);
                const float en = fmaf(e, rt, lf[k]);
                lf[k] = en;
                const int c = ch.chain_of[k];
                aPf[c] = fmaf(R, en, aPf[c]); aQf[c] = fmaf(X, en, aQf[c]);
            }
            for (int c = ch.n - 1; c >= 0; --c) {
                UPf[c] = aPf[c]; UQf[c] = aQf[c];
                for (int d = c + 1; d < ch.n; ++d) if ((ch.child[c] >> d) & 1u) { UPf[c] = UPf[c] + UPf[d]; UQf[c] = UQf[c] + UQf[d]; }
            }
            ++it;
        }
        for (int k = 0; k < NL; ++k) ell[k] = (double)lf[k];
        for (int c = 0; c < MAXCH; ++c) { UP[c] = (double)UPf[c]; UQ[c] = (double)UQf[c]; }
    }
    while (it < max_iter) {
        ++it;
        conv = 1;
        for (int c = 0; c < MAXCH; ++c) aP[c] = aQ[c] = 0.0;
        /* a chain's lines are consecutive lanes, so one carried (W_P, W_Q) pair serves every chain */
        double wP = 0.0, wQ = 0.0;
        for (int k = 0; k < t->nl; ++k) {
            double P, Q;
            line_t(t, &ch, k, SP, SQ, ell[k], UP, UQ, &wP, &wQ, v, &P, &Q);
            double vk = v[k];
            if (sqv_bad(vk)) bad = 1;
            double s = P * P;
            s = fma(Q, Q, s);
            double e = fma(-vk, ell[k], s);          /* residual of the current row at the old current */
            double d = 1.0 - vk, rt = 2.0 - vk;
            rt = fma(d, rt, 1.0);                    /* 1 + d + d^2 = (1 - d^3) / v */
            double en = fma(e, rt, ell[k]);
            if (!(hi_abs(e) < hi_abs(tol))) conv = 0;
            ell[k] = en;
            int c = ch.chain_of[k];
            aP[c] = fma(t->R[k], en, aP[c]); aQ[c] = fma(t->X[k], en, aQ[c]);
        }
        for (int c = ch.n - 1; c >= 0; --c) {
            UP[c] = aP[c]; UQ[c] = aQ[c];
            for (int d = c + 1; d < ch.n; ++d) if ((ch.child[c] >> d) & 1u) { UP[c] = UP[c] + UP[d]; UQ[c] = UQ[c] + UQ[d]; }
        }
        if (bad || conv) break;
    }
    {
        double wP = 0.0, wQ = 0.0;
        for (int k = 0; k < t->nl; ++k) {
            line_t(t, &ch, k, SP, SQ, ell[k], UP, UQ, &wP, &wQ, v, &o->P[k], &o->Q[k]);
            if (sqv_bad(v[k])) bad = 1;
        }
    }
    for (int k = 0; k < NL; ++k) { o->v[k] = v[k]; o->ell[k] = ell[k]; }
    o->iters = it; o->ok = conv && !bad;
}

static void sweep(const FoNet* t, const double* p, const double* q, double tol, int max_iter, Sweep* o) {
    if (t->variant == 0) sweep_t(t, p, q, tol, max_iter, o);
    else sweep_w(t, p, q, tol, max_iter, o);
}

/* Batched power flow: p/q [n][nl] bus order -> V [n][nb], Pl/Ql/Isq [n][nl] (may be NULL). */
void fo_power_flow(const FoNet* t, double tol, int max_iter, int64_t n, const double* p, const double* q,
                   double* V, double* Pl, double* Ql, double* Isq, int32_t* iters, uint8_t* fail) {
    const int nl = t->nl, nb = t->nb;
#pragma omp parallel for schedule(static)
    for (int64_t e = 0; e < n; ++e) {
        double pl[NL] = {0}, ql[NL] = {0};
        Sweep s;
        for (int k = 0; k < nl; ++k) { pl[k] = p[e * nl + t->col[k]]; ql[k] = q[e * nl + t->col[k]]; }
        sweep(t, pl, ql, tol, max_iter, &s);
        V[e * nb] = 1.0;
        for (int k = 0; k < nl; ++k) {
            int c = t->col[k];
            V[e * nb + c + 1] = sqrt(s.v[k]);
            if (Pl) Pl[e * nl + c] = s.P[k];
            if (Ql) Ql[e * nl + c] = s.Q[k];
            if (Isq) Isq[e * nl + c] = s.ell[k];
        }
        if (iters) iters[e] = s.iters;
        if (fail) fail[e] = s.ok ? 0 : 1;
    }
}

static double clipd(double x, double lo, double hi) { double t = x > lo ? x : lo; return t < hi ? t : hi; }

typedef struct { double pred, ch, dis, qpv; } Setp;

/* x / d with r = RN(1/d): q0 = x r, rem = x - q0 d (exact), q = q0 + rem r -- the correctly rounded
 * quotient (Markstein), which is what the kernels evaluate instead of a division subroutine */
static double div_const(double x, double d, double r) {
    double q0 = x * r, rem = fma(-q0, d, x);
    return fma(rem, r, q0);
}

static void ess_clip(const FoNet* c, double* ch_, double* dis_, double e_now) {
    double ch = clipd(*ch_, 0.0, c->p_ch_max), dis = clipd(*dis_, 0.0, c->p_dis_max);
    const double inv_eta_dis = 1.0 / c->eta_dis, inv_eta_ch = 1.0 / c->eta_ch;
    double e_next = (e_now + c->eta_ch * ch) - inv_eta_dis * dis;
    if (e_next > c->e_max) {
        double excess = e_next - c->e_max, tt = div_const(excess, c->eta_ch, inv_eta_ch);
        if (ch > tt) ch = ch - tt;
        else { dis = dis + (excess - ch * c->eta_ch) * c->eta_dis; ch = 0.0; }
    } else if (e_next < c->e_min) {
        double lack = c->e_min - e_next, tt = lack * c->eta_dis;
        if (dis > tt) dis = dis - tt;
        else { ch = ch + div_const(lack - div_const(dis, c->eta_dis, inv_eta_dis), c->eta_ch, inv_eta_ch); dis = 0.0; }
    }
    *ch_ = clipd(ch, 0.0, c->p_ch_max); *dis_ = clipd(dis, 0.0, c->p_dis_max);
}

static Setp setpoints(const FoNet* c, int scale, const double* a, double pload, double ppv, double e_clip) {
    double pct, ch, dis, qpv;
    if (scale) {
        pct = c->mpr * a[0]; ch = c->p_ch_max * a[1]; dis = c->p_dis_max * a[2];
        double lim = c->kappa * ppv, lo = -lim;
        qpv = clipd(lo + a[3] * (lim - lo), lo, lim);
    } else { pct = a[0]; ch = a[1]; dis = a[2]; qpv = a[3]; }
    pct = clipd(pct, 0.0, c->mpr);
    if (ch > 0.0 && dis > 0.0) { if (ch > dis) { ch = ch - dis; dis = 0.0; } else { dis = dis - ch; ch = 0.0; } }
    ess_clip(c, &ch, &dis, e_clip);
    Setp s; s.pred = pload * pct; s.ch = ch; s.dis = dis; s.qpv = qpv;
    return s;
}

/* Plain per-env state, struct of arrays. */
typedef struct {
    int64_t n;
    double *E_init, *E_cur;      /* [n][na] */
    double* cum;                 /* [n] */
    int32_t *start, *steps, *episode, *hist_n;
    double* V;                   /* [n][nb] */
    double* setp;                /* [n][4][na] */
    uint64_t* vmask; int32_t *vcount, *flags, *iters; uint32_t* lmask;
    double *pfl, *qfl, *isq;     /* [n][nl] */
} FoState;

/* butterfly sum: after rounds d=16,8,4,2,1 every lane holds the same value */
static double xor_sum32(const double* x) {
    double s[NL], n2[NL];
    memcpy(s, x, sizeof(s));
    for (int d = 16; d >= 1; d >>= 1) {
        for (int k = 0; k < NL; ++k) n2[k] = s[k] + s[k ^ d];
        memcpy(s, n2, sizeof(s));
    }
    return s[0];
}

static void philox(uint32_t c[4], uint32_t k0, uint32_t k1) {
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0, n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1, n3 = (uint32_t)p0;
        c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}
static double u53(uint32_t a, uint32_t b) {
    return (double)(((uint64_t)(a >> 5) << 26) | (uint64_t)(b >> 6)) * (1.0 / 9007199254740992.0);
}

/* Draws of one env for fp_reset_random: start, e0[na], a0[4*na]. */
void fo_random_draw(const FoNet* c, uint64_t seed, int64_t gid, int32_t episode, int32_t start_range,
                    int32_t* start, double* e0, double* a0) {
    double u0[16], u1[16];
    for (int b = 0; b < 16; ++b) {
        uint32_t ctr[4] = {(uint32_t)gid, (uint32_t)((uint64_t)gid >> 32), (uint32_t)episode, (uint32_t)b};
        philox(ctr, (uint32_t)seed, (uint32_t)(seed >> 32));
        u0[b] = u53(ctr[0], ctr[1]); u1[b] = u53(ctr[2], ctr[3]);
    }
    double lo = 0.9 * (c->e_max / 2), hi = 1.1 * (c->e_max / 2);
    *start = (int32_t)(u0[15] * (double)start_range);
    for (int i = 0; i < c->na; ++i) {
        e0[i] = lo + (hi - lo) * u0[10 + i];
        a0[4 * i + 0] = u0[2 * i]; a0[4 * i + 1] = u1[2 * i];
        a0[4 * i + 2] = u0[2 * i + 1]; a0[4 * i + 3] = u1[2 * i + 1];
    }
}

/* One env, shared by reset (is_reset=1) and step.  actions: 4*na doubles. */
static void env_core(const FoNet* c, const double* P, const double* Q, const double* PV, const double* price,
                     FoState* s, int64_t e, int is_reset, const double* act, int inject,
                     double* reward, uint8_t* done, double* info) {
    const int nl = c->nl, nb = c->nb, na = c->na;
    int32_t steps = is_reset ? 1 : s->steps[e];
    /* quirk Q1; an env stepped on past `done` without a reset stays on the last row of its slice (episode_limit +
       history + 1 rows), as the kernels do (row_in_force) */
    const int max_off = c->episode_limit + c->history;
    const int64_t row = (int64_t)s->start[e] + ((!is_reset && steps > 1) ? (steps - 1 < max_off ? steps - 1 : max_off) : 1);
    double pl[NL] = {0}, ql[NL] = {0};
    Setp sp[8];
    for (int k = 0; k < nl; ++k) { pl[k] = P[row * nl + c->col[k]]; ql[k] = Q[row * nl + c->col[k]]; }
    const double lam = price[row];
    for (int i = 0; i < na; ++i) {
        double pload = P[row * nl + c->agent_col[i]], ppv = PV[row * na + i];
        double e_clip = is_reset ? s->E_init[e * na + i] : s->E_cur[e * na + i];
        sp[i] = setpoints(c, is_reset || !c->raw_actions, act + 4 * i, pload, ppv, e_clip);
        int k = c->agent_lane[i];
        pl[k] = (((pload - sp[i].pred) - ppv) + sp[i].ch) - sp[i].dis;
        ql[k] = ql[k] - sp[i].qpv;
    }
    Sweep sw;
    sweep(c, pl, ql, c->pf_tol, c->pf_max_iter, &sw);
    int ok = sw.ok && !inject;
    /* a NaN action: np.clip keeps it, the reference's NLP gets a NaN injection and its solve raises (:314-337) */
    if (!is_reset) for (int k = 0; k < 4 * na; ++k) if (act[k] != act[k]) ok = 0;
    double e_next[8];
    const double inv_eta_dis = 1.0 / c->eta_dis;
    for (int i = 0; i < na; ++i) {
        e_next[i] = s->E_init[e * na + i] + c->delta_t * (c->eta_ch * sp[i].ch - inv_eta_dis * sp[i].dis);
        if (e_next[i] < c->e_next_lb) ok = 0;
    }
    double V[NL];
    for (int k = 0; k < NL; ++k) V[k] = sqrt(sw.v[k]);
    if (ok) {
        s->V[e * nb] = 1.0;
        for (int k = 0; k < nl; ++k) s->V[e * nb + c->col[k] + 1] = V[k];
        if (s->pfl) for (int k = 0; k < nl; ++k) {
            s->pfl[e * nl + c->col[k]] = sw.P[k]; s->qfl[e * nl + c->col[k]] = sw.Q[k]; s->isq[e * nl + c->col[k]] = sw.ell[k];
        }
    } else if (!is_reset) {
        for (int k = 0; k < nl; ++k) V[k] = s->V[e * nb + c->col[k] + 1];
        for (int i = 0; i < na; ++i) {
            sp[i].pred = s->setp[e * 4 * na + 0 * na + i]; sp[i].ch = s->setp[e * 4 * na + 1 * na + i];
            sp[i].dis = s->setp[e * 4 * na + 2 * na + i]; sp[i].qpv = s->setp[e * 4 * na + 3 * na + i];
        }
    }
    double vterm[NL] = {0};
    uint32_t vm = 0, lm = 0;
    for (int k = 0; k < nl; ++k) {
        double over = V[k] - c->v_max, under = c->v_min - V[k];
        if (over > 0.0 || under > 0.0) { vm |= 1u << c->col[k]; vterm[k] = c->voltage_coeff * (over > under ? over : under); }
        if (ok && sw.ell[k] > c->imax2[k]) lm |= 1u << c->col[k];
    }
    const double s_over = 1.0 - c->v_max, s_under = c->v_min - 1.0;
    const int slack_viol = (s_over > 0.0 || s_under > 0.0);
    const double slack_pen = slack_viol ? c->voltage_coeff * (s_over > s_under ? s_over : s_under) : 0.0;
    s->vmask[e] = ((uint64_t)vm << 1) | (uint64_t)slack_viol;
    s->vcount[e] = __builtin_popcount(vm) + slack_viol;
    s->lmask[e] = lm; s->iters[e] = sw.iters;
    if (is_reset) {
        for (int i = 0; i < na; ++i) {
            s->E_cur[e * na + i] = ok ? e_next[i] : s->E_init[e * na + i];
            s->setp[e * 4 * na + 0 * na + i] = sp[i].pred; s->setp[e * 4 * na + 1 * na + i] = sp[i].ch;
            s->setp[e * 4 * na + 2 * na + i] = sp[i].dis; s->setp[e * 4 * na + 3 * na + i] = sp[i].qpv;
        }
        s->cum[e] = 0.0; s->steps[e] = 1; s->hist_n[e] = 0; s->episode[e] += 1;
        s->flags[e] = ok ? 0 : 4;
        return;
    }
    double vpen;
    if (c->variant == 0) { vpen = 0.0; for (int k = 0; k < nl; ++k) vpen = vpen + vterm[k]; vpen = vpen + slack_pen; }
    else vpen = xor_sum32(vterm) + slack_pen;
    double rev = lam * sp[0].pred, der = c->pv_cost * sp[0].qpv, ess = c->ess_cost * (sp[0].ch + sp[0].dis),
           disc = c->discomfort_coeff * (sp[0].pred * sp[0].pred);
    for (int i = 1; i < na; ++i) {
        rev = rev + lam * sp[i].pred; der = der + c->pv_cost * sp[i].qpv;
        ess = ess + c->ess_cost * (sp[i].ch + sp[i].dis); disc = disc + c->discomfort_coeff * (sp[i].pred * sp[i].pred);
    }
    double r = (((rev - der) - ess) - disc) - vpen;
    if (info) {
        double* o = info + e * 8;
        o[0] = r; o[1] = rev; o[2] = der; o[3] = ess; o[4] = disc; o[5] = vpen; o[6] = s->cum[e]; o[7] = ok ? 0.0 : 1.0;
    }
    if (!ok) r = r - c->fail_penalty;
    int steps_new = steps + 1;
    int dn = (steps_new >= c->episode_limit) || !ok;
    reward[e] = r; done[e] = (uint8_t)dn;
    s->cum[e] = s->cum[e] + r; s->steps[e] = steps_new;
    s->flags[e] = (dn ? 1 : 0) | (ok ? 0 : 2);
    for (int i = 0; i < na; ++i) {
        double ec = ok ? e_next[i] : s->E_cur[e * na + i];
        s->E_cur[e * na + i] = ec; s->E_init[e * na + i] = ec;
        if (ok) {
            s->setp[e * 4 * na + 0 * na + i] = sp[i].pred; s->setp[e * 4 * na + 1 * na + i] = sp[i].ch;
            s->setp[e * 4 * na + 2 * na + i] = sp[i].dis; s->setp[e * 4 * na + 3 * na + i] = sp[i].qpv;
        }
    }
}

/* reset: start[n], e0[n][na], a0[n][4na]; mask may be NULL */
void fo_env_reset(const FoNet* c, const double* P, const double* Q, const double* PV, const double* price,
                  FoState* s, const int32_t* start, const double* e0, const double* a0, const uint8_t* mask) {
    const int na = c->na;
#pragma omp parallel for schedule(static)
    for (int64_t e = 0; e < s->n; ++e) {
        if (mask && !mask[e]) continue;
        s->start[e] = start[e];
        for (int i = 0; i < na; ++i) s->E_init[e * na + i] = e0[e * na + i];
        env_core(c, P, Q, PV, price, s, e, 1, a0 + e * 4 * na, 0, NULL, NULL, NULL);
    }
}

void fo_env_reset_random(const FoNet* c, const double* P, const double* Q, const double* PV, const double* price,
                         FoState* s, uint64_t seed, int64_t env_offset, int32_t start_range, const uint8_t* mask) {
    const int na = c->na;
#pragma omp parallel for schedule(static)
    for (int64_t e = 0; e < s->n; ++e) {
        if (mask && !mask[e]) continue;
        double e0[8], a0[32];
        int32_t st;
        fo_random_draw(c, seed, env_offset + e, s->episode[e], start_range, &st, e0, a0);
        s->start[e] = st;
        for (int i = 0; i < na; ++i) s->E_init[e * na + i] = e0[i];
        env_core(c, P, Q, PV, price, s, e, 1, a0, 0, NULL, NULL, NULL);
    }
}

/* step: actions [n][4na] fp64 (caller widens fp32 exactly); inject/mask may be NULL */
void fo_env_step(const FoNet* c, const double* P, const double* Q, const double* PV, const double* price,
                 FoState* s, const double* actions, const uint8_t* inject, const uint8_t* mask,
                 double* reward, uint8_t* done, double* info) {
    const int na = c->na;
#pragma omp parallel for schedule(static)
    for (int64_t e = 0; e < s->n; ++e) {
        if (mask && !mask[e]) continue;
        env_core(c, P, Q, PV, price, s, e, 0, actions + e * 4 * na, inject ? inject[e] : 0, reward, done, info);
    }
}

/* OpenMP worker threads the batched entry points will use (bench.py reports it as `cores`). */
#ifdef _OPENMP
#include <omp.h>
int fo_threads(void) { return omp_get_max_threads(); }
void fo_set_threads(int n) { if (n > 0) omp_set_num_threads(n); }
#else
int fo_threads(void) { return 1; }
void fo_set_threads(int n) { (void)n; }
#endif

int fo_sizeof_net(void) { return (int)sizeof(FoNet); }
int fo_sizeof_state(void) { return (int)sizeof(FoState); }
