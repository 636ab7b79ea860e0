// flex_env_math.cuh -- per-agent arithmetic of the env step, shared by the warp-per-env and the
// thread-per-env kernels (action scaling, ESS anti-simultaneity and energy clipping).
#pragma once
#include "flex_common.cuh"

// Setpoints of one agent (executed by the agent's lane).
struct Setpoint { double pred, ch, dis, qpv; };

// x / d for a constant divisor with r = RN(1 / d): one multiplication and two fused
// multiply-adds give the CORRECTLY ROUNDED quotient (Markstein: q0 = x r, rem = x - q0 d exactly,
// q = q0 + rem r), i.e. the bits of the reference's Python `x / d`, without the division
// subroutine and its branches (checked against true division on 4e8 values; mirrored in
// oracle/c/flex_oracle.c).
__device__ __forceinline__ double div_const(double x, double d, double r) {
    const double q0 = x * r;
    const double rem = fma(-q0, d, x);
    return fma(rem, r, q0);
}

// The clip of the action parsing: NanClip = false for the step, reset and preview kernels (clipd), true for the safety
// layer, whose NaN proposals must stay NaN as under numpy.clip (clip_np).
template <bool NanClip>
__device__ __forceinline__ double clip_act(double x, double lo, double hi) {
    return NanClip ? clip_np(x, lo, hi) : clipd(x, lo, hi);
}

// flexibility_provision_env.py:628-661 (no delta_t here -- quirk Q3).  Branch-free: both
// candidate corrections are evaluated and selected, so the 32 envs of a warp never diverge.
template <bool NanClip = false>
__device__ __forceinline__ void ess_energy_clip(const DevCfg& c, double& ch, double& dis, double e_now) {
    ch = clip_act<NanClip>(ch, 0.0, c.p_ch_max);
    dis = clip_act<NanClip>(dis, 0.0, c.p_dis_max);
    const double e_next = (e_now + c.eta_ch * ch) - c.inv_eta_dis * dis;
    const bool over = e_next > c.e_max, under = !over && (e_next < c.e_min);
    // e_next > e_max (:637-646)
    const double excess = e_next - c.e_max;
    const double t = div_const(excess, c.eta_ch, c.inv_eta_ch);
    const bool o1 = ch > t;
    const double ch_o = o1 ? (ch - t) : 0.0;
    const double dis_o = o1 ? dis : (dis + (excess - ch * c.eta_ch) * c.eta_dis);
    // e_next < e_min (:647-656)
    const double lack = c.e_min - e_next;
    const double t2 = lack * c.eta_dis;
    const bool u1 = dis > t2;
    const double dis_u = u1 ? (dis - t2) : 0.0;
    const double ch_u = u1 ? ch : (ch + div_const(lack - div_const(dis, c.eta_dis, c.inv_eta_dis), c.eta_ch, c.inv_eta_ch));
    ch = over ? ch_o : (under ? ch_u : ch);
    dis = over ? dis_o : (under ? dis_u : dis);
    ch = clip_act<NanClip>(ch, 0.0, c.p_ch_max);
    dis = clip_act<NanClip>(dis, 0.0, c.p_dis_max);
}

// :262-293 (step) / :113-130 (reset): raw action -> applied setpoints, everything that does not
// need the building's load: `pred` returns the clipped reduction FRACTION (:676-677).  NanClip: see clip_act.
template <bool NanClip = false>
__device__ __forceinline__ Setpoint apply_actions_frac(const DevCfg& c, bool scale, double a0, double a1,
                                                       double a2, double a3, double ppv, double e_clip) {
    double pct, ch, dis, qpv;
    if (scale) {
        pct = c.mpr * a0;                                   // :278
        ch = c.p_ch_max * a1;                               // :279
        dis = c.p_dis_max * a2;                             // :280
        double lim = c.kappa * ppv;                         // :623
        double lo = -lim;
        qpv = clip_act<NanClip>(lo + a3 * (lim - lo), lo, lim);   // :626
    } else {                                                // 'safemaddpg' branch :268-274
        pct = a0; ch = a1; dis = a2; qpv = a3;
    }
    pct = clip_act<NanClip>(pct, 0.0, c.mpr);               // :676-677
    {                                                       // :663-674, branch-free
        const bool both = (ch > 0.0) && (dis > 0.0), gt = ch > dis;
        const double ch2 = gt ? (ch - dis) : 0.0, dis2 = gt ? 0.0 : (dis - ch);
        ch = both ? ch2 : ch; dis = both ? dis2 : dis;
    }
    ess_energy_clip<NanClip>(c, ch, dis, e_clip);           // :289-290
    Setpoint s;
    s.pred = pct;
    s.ch = ch; s.dis = dis; s.qpv = qpv;
    return s;
}

__device__ __forceinline__ Setpoint apply_actions(const DevCfg& c, bool scale, double a0, double a1,
                                                  double a2, double a3, double pload, double ppv,
                                                  double e_clip) {
    Setpoint s = apply_actions_frac(c, scale, a0, a1, a2, a3, ppv, e_clip);
    s.pred = pload * s.pred;                                // :293
    return s;
}
