"""The safety layer's fp64 restatement over a whole batch, for checking both safety kernels on every row.

  parse_actions    safety_ref.parse_actions over [N, na, 4]: numpy.clip semantics (a NaN stays NaN) and env_ref's
                   operation order, so that it equals the scalar oracle bit for bit (tests/test_oracle_safety_batch.py)
  project_rowsum   safety_ref.project_closed_form over [N, na], the same segment walk, bit for bit
  project_affine   safety_affine_ref.project_affine over [N]: one GEMV classifies every env; an env whose V(y0) is inside
                   the limits by more than the GEMV's rounding is returned as proposed, one with a non-finite V(y0) is
                   left unprojected (the scalar restatement's contract), every other env runs the scalar restatement,
                   in worker processes when an AffinePool is given

Inputs come from env.get_state(torch.float64): P, Q in bus order (0 at the slack bus), PV and E of the agents at the row
in force -- what the kernels read.  No torch here: AffinePool's workers are spawned and import only numpy and the oracle.
"""
import multiprocessing
import os
from concurrent.futures import ProcessPoolExecutor
from math import acos, tan

import numpy as np

from oracle import safety_affine_ref, safety_ref

W_SLACK = safety_ref.W_SLACK


def split_state(state, nb, na):
    """fp64 get_state rows [N, P(nb) Q(nb) Ppv(na) V(nb) price E(na)] -> P [N, nb], Q [N, nb], PV [N, na], E [N, na]."""
    s = np.asarray(state, dtype=np.float64)
    return s[:, :nb], s[:, nb:2 * nb], s[:, 2 * nb:2 * nb + na], s[:, 3 * nb + na + 1:3 * nb + 2 * na + 1]


def parse_actions(args, pv, e_now, actions):
    """safemaddpg.py:143-174 for every (env, agent): raw actions [N, na, 4], PV and ESS energy [N, na] -> the proposal
    y0 [N, na, 4] = (power-reduction fraction, charge, discharge, q_pv) in env_ref's operation order."""
    a = np.asarray(actions, dtype=np.float64)
    pv = np.asarray(pv, dtype=np.float64); e_now = np.asarray(e_now, dtype=np.float64)
    mpr, pch, pdis = args["max_power_reduction"], args["p_ch_max"], args["p_dis_max"]
    eta_ch, eta_dis, e_min, e_max = args["eta_ch"], args["eta_dis"], args["e_min"], args["e_max"]
    with np.errstate(all="ignore"):
        pct = mpr * a[..., 0]
        ch = pch * a[..., 1]
        dis = pdis * a[..., 2]
        c = tan(acos(args["cos_phi_max"])) * pv                                # _scale_and_clip_q_pv
        qpv = np.clip(-c + a[..., 3] * (c - (-c)), -c, c)
        pct = np.clip(pct, 0, mpr)                                             # clip_percentage_reduction
        both = (ch > 0) & (dis > 0)                                            # adjust_ess_actions
        gt = ch > dis
        ch, dis = (np.where(both, np.where(gt, ch - dis, 0.0), ch), np.where(both, np.where(gt, 0.0, dis - ch), dis))
        ch = np.clip(ch, 0, pch)                                               # _clip_power_charging_discharging
        dis = np.clip(dis, 0, pdis)
        e_next = e_now + eta_ch * ch - (1 / eta_dis) * dis
        over = e_next > e_max
        under = ~over & (e_next < e_min)
        excess = e_next - e_max
        o1 = ch > excess / eta_ch
        ch_o = np.where(o1, ch - excess / eta_ch, 0.0)
        dis_o = np.where(o1, dis, dis + (excess - ch * eta_ch) * eta_dis)
        lack = e_min - e_next
        u1 = dis > lack * eta_dis
        dis_u = np.where(u1, dis - lack * eta_dis, 0.0)
        ch_u = np.where(u1, ch, ch + (lack - dis / eta_dis) / eta_ch)
        ch = np.where(over, ch_o, np.where(under, ch_u, ch))
        dis = np.where(over, dis_o, np.where(under, dis_u, dis))
        ch = np.clip(ch, 0, pch)
        dis = np.clip(dis, 0, pdis)
    return np.stack([pct, ch, dis, qpv], axis=-1)


def rowsum_prediction(y0, Pd, Qd, sP, sQ, b):
    """V(y0) of project_closed_form for every (env, agent), in its operation order (the kernel fuses the sQ term)."""
    with np.errstate(all="ignore"):
        return sP * (Pd * (1.0 - y0[..., 0]) + y0[..., 1] - y0[..., 2]) + sQ * (Qd + y0[..., 3]) + b


def project_rowsum(y0, Pd, Qd, sP, sQ, b, v_min, v_max, w=W_SLACK):
    """project_closed_form for every (env, agent): y0 [N, na, 4]; Pd, Qd [N, na] the agents' own demands; sP, sQ, b [na]
    the row sums at the agents' buses.  Returns (y [N, na, 4], slack [N, na], lam [N, na])."""
    y0 = np.asarray(y0, dtype=np.float64)
    V0 = rowsum_prediction(y0, Pd, Qd, sP, sQ, b)
    with np.errstate(all="ignore"):
        low, high = V0 < v_min, V0 > v_max
        delta = np.where(low, v_min - V0, np.where(high, V0 - v_max, 0.0))
        sgn = np.where(low, 1.0, -1.0)
        a = np.stack([sgn * (-sP * Pd), sgn * np.broadcast_to(sP, Pd.shape), sgn * (-np.broadcast_to(sP, Pd.shape)),
                      sgn * np.broadcast_to(sQ, Pd.shape)], axis=-1)
        t = np.where(a[..., :3] < 0.0, 2.0 * y0[..., :3] / -a[..., :3], np.inf)     # breakpoint of a falling variable
        brk = np.sort(t, axis=-1)

        def slope(lam):
            s = a[..., 3] * a[..., 3] / 2.0
            for i in range(3):
                on = (a[..., i] > 0.0) | ((a[..., i] < 0.0) & (lam < t[..., i]))
                s = np.where(on, s + a[..., i] * a[..., i] / 2.0, s)
            return s
        lam = np.zeros_like(V0); gain = np.zeros_like(V0)
        live = low | high
        for j in range(4):
            nxt = np.minimum(brk[..., j], w) if j < 3 else np.full_like(V0, w)
            go = live & ~(nxt <= lam)
            s = slope(lam)
            close = go & (s > 0.0) & (gain + s * (nxt - lam) >= delta)
            lam_c = lam + (delta - gain) / s
            gain_a = gain + s * (nxt - lam)
            adv = go & ~close
            lam = np.where(close, lam_c, np.where(adv, nxt, lam))
            gain = np.where(close, delta, np.where(adv, gain_a, gain))
            live = live & ~close & ~(adv & (lam >= w))
        y = y0.copy()
        for i in range(3):
            v = y0[..., i] + 0.5 * lam * a[..., i]
            y[..., i] = np.where(0.0 > v, 0.0, v)                                 # Python's max(v, 0.0)
        y[..., 3] = y0[..., 3] + 0.5 * lam * a[..., 3]
        moved = low | high
        y = np.where(moved[..., None], y, y0)
        slack = np.where(moved, np.maximum(0.0, delta - gain), 0.0)
        lam = np.where(moved, lam, 0.0)
    return y, slack, lam


def affine_prediction(y0, Pd, Qd, agent_bus, A, c):
    """V(y0) for every env (one GEMV): y0 [N, na, 4]; Pd, Qd [N, nb] bus order.  Also |A| |x| + |c|, the scale of the
    rounding error of any summation order."""
    P = np.array(Pd, dtype=np.float64); Q = np.array(Qd, dtype=np.float64)
    with np.errstate(all="ignore"):
        P[:, agent_bus] = Pd[:, agent_bus] * (1.0 - y0[..., 0]) + y0[..., 1] - y0[..., 2]
        Q[:, agent_bus] = Qd[:, agent_bus] + y0[..., 3]
        x = np.empty((P.shape[0], 2 * P.shape[1])); x[:, 0::2] = P; x[:, 1::2] = Q
        return x @ A.T + c, np.abs(x) @ np.abs(A).T + np.abs(c)


def _affine_rows(job):
    y0, Pd, Qd, agent_bus, A, c, v_min, v_max, w = job
    out = [safety_affine_ref.project_affine(y0[i], Pd[i], Qd[i], agent_bus, A, c, v_min, v_max, w) for i in range(len(y0))]
    return (np.stack([o[0] for o in out]), np.stack([o[1] for o in out]), np.array([o[2] for o in out], dtype=np.int32))


class AffinePool:
    """Spawned worker processes for the scalar restatement (no torch, no CUDA in them).  A context manager: the workers
    end with the block."""

    def __init__(self, workers=None):
        n = workers or len(os.sched_getaffinity(0))
        self.workers = max(1, min(32, n))
        self.ex = ProcessPoolExecutor(self.workers, mp_context=multiprocessing.get_context("spawn"))

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.ex.shutdown(wait=True, cancel_futures=True)

    def map(self, jobs):
        return list(self.ex.map(_affine_rows, jobs))


DV_ROUND = 1e-12            # an env whose V(y0) is this close (relative to |A| |x| + |c|) to a limit runs the restatement


def project_affine(y0, Pd, Qd, agent_bus, A, c, v_min, v_max, w=W_SLACK, pool=None, chunk=64):
    """project_affine for every env: y0 [N, na, 4]; Pd, Qd [N, nb].  Returns (y [N, na, 4], slack [N, nb], status [N],
    n_scalar: the envs the scalar restatement ran)."""
    y0 = np.asarray(y0, dtype=np.float64); A = np.asarray(A, dtype=np.float64); c = np.asarray(c, dtype=np.float64)
    agent_bus = np.asarray(agent_bus, dtype=np.int64)
    N, nb = Pd.shape
    V, scale = affine_prediction(y0, Pd, Qd, agent_bus, A, c)
    tol = DV_ROUND * np.maximum(1.0, scale)
    finite = np.isfinite(V).all(axis=1)
    inside = ((V >= v_min + tol) & (V <= v_max - tol)).all(axis=1)
    run = np.flatnonzero(finite & ~inside)
    y, slack, status = y0.copy(), np.zeros((N, nb)), np.zeros(N, dtype=np.int32)
    if len(run):
        jobs = [(y0[r], Pd[r], Qd[r], agent_bus, A, c, v_min, v_max, w) for r in np.array_split(run, -(-len(run) // chunk))]
        res = pool.map(jobs) if pool is not None and len(jobs) > 1 else [_affine_rows(j) for j in jobs]
        y[run] = np.concatenate([r[0] for r in res]); slack[run] = np.concatenate([r[1] for r in res])
        status[run] = np.concatenate([r[2] for r in res])
    return y, slack, status, len(run)


def bits_moved(y, y0):
    """Per (env, agent): any of the four values changed, compared as bits (an untouched NaN has not moved)."""
    return (np.asarray(y, dtype=np.float64).view(np.int64) != np.asarray(y0, dtype=np.float64).view(np.int64)).any(axis=-1)
