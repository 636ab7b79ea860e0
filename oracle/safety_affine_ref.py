"""fp64 restatement of the safety layer against the full fitted voltage map (oracle side): the QP of
madrl/models/safemaddpg.py:176-299 with V = A [P_1, Q_1, ..., P_nb, Q_nb] + c, the regressor as it was trained, in place of
the reference's row-sum reading (SURVEY 3.6, oracle/safety_ref.py).  What fp_safety_project_affine computes.

TEST INFRASTRUCTURE (see oracle/__init__.py).  The reference never poses this problem (it only evaluates the row sums), so
there is nothing of the reference to pin it to; what pins it instead:

  solve_affine_qp   the 86-variable QP posed as safety_ref.solve_reference_qp poses the reference's model -- all 20 action
                    variables, P_net / Q_net of every bus, nb lower and nb upper slacks priced at w -- with the prediction
                    map as a parameter (posed_qp), handed to the same generic solver (scipy trust-constr).  With the
                    row-sum map posed_qp is solve_reference_qp (tests/test_oracle_safety_affine.py checks this).
  project_affine    the active-set method the CUDA kernel runs, step for step; it must agree with solve_affine_qp, with
                    safety_ref.project_closed_form on a row-sum map, and pass a KKT perturbation test.
"""
import numpy as np

from .safety_ref import W_SLACK


def solve_affine_qp(y0, Pd, Qd, is_building, A, c, v_min, v_max, w=W_SLACK):
    """The same QP with the full fitted map V = A [P_1, Q_1, ..., P_nb, Q_nb] + c (A [nb, 2 nb], interleaved inputs as the
    regressor was trained) in place of the reference's row sums: every bus depends on every building's actions."""
    A = np.asarray(A, dtype=np.float64); c = np.asarray(c, dtype=np.float64)

    def vmap(P, Q):
        x = np.empty(2 * len(P)); x[0::2] = P; x[1::2] = Q
        return A @ x + c
    return posed_qp(y0, Pd, Qd, is_building, vmap, v_min, v_max, w)


def posed_qp(y0, Pd, Qd, is_building, vmap, v_min, v_max, w):
    """safety_ref.solve_reference_qp's posing with the prediction as a parameter: all 4 nb_buildings action variables,
    nb lower and nb upper slacks, vmap(P_net [nb], Q_net [nb]) -> V [nb], handed to scipy trust-constr.
    Returns (optimal [nb_buildings, 4], scipy result)."""
    from scipy.optimize import minimize
    nbld, nbus = y0.shape[0], len(Pd)
    nv = 4 * nbld + 2 * nbus                                   # actions, slack_lower[33], slack_upper[33]
    # scale the variables so that the solver sees O(1) numbers: actions and slacks in units of 1e-3
    S = 1e-3

    def vpred(z):
        y = z[:4 * nbld].reshape(nbld, 4) * S
        P = Pd.copy(); Q = Qd.copy()
        for n in range(nbus):
            k = is_building[n]
            if k >= 0:
                P[n] = Pd[n] * (1.0 - y[k, 0]) + y[k, 1] - y[k, 2]
                Q[n] = Qd[n] + y[k, 3]
        return vmap(P, Q)

    # V_pred is affine in z: V = V(0) + J z  (exact: probe the columns)
    from scipy.optimize import Bounds, LinearConstraint
    v_at0 = vpred(np.zeros(nv))
    J = np.zeros((nbus, nv))
    for j in range(4 * nbld):
        e = np.zeros(nv); e[j] = 1.0
        J[:, j] = vpred(e) - v_at0
    A_lo = J.copy(); A_lo[:, 4 * nbld:4 * nbld + nbus] += S * np.eye(nbus)          # V + s_lo >= v_min
    A_up = -J.copy(); A_up[:, 4 * nbld + nbus:] += S * np.eye(nbus)                  # -V + s_up >= -v_max
    A = np.vstack([A_lo, A_up]) / S
    lb = np.concatenate([v_min - v_at0, v_at0 - v_max]) / S
    lo = np.full(nv, -np.inf); lo[4 * nbld:] = 0.0
    for k in range(nbld):
        lo[4 * k:4 * k + 3] = 0.0
    grad_lin = np.zeros(nv); grad_lin[4 * nbld:] = w * S / S ** 2
    y0s = y0.reshape(-1) / S

    def obj(z):
        d = z[:4 * nbld] - y0s
        return float(d @ d + grad_lin @ z)

    def jac(z):
        g = grad_lin.copy(); g[:4 * nbld] += 2.0 * (z[:4 * nbld] - y0s)
        return g

    def hess(z):
        H = np.zeros((nv, nv)); H[np.arange(4 * nbld), np.arange(4 * nbld)] = 2.0
        return H
    z0 = np.zeros(nv)
    z0[:4 * nbld] = y0s
    v0 = vpred(z0)
    z0[4 * nbld:4 * nbld + nbus] = np.maximum(0.0, v_min - v0) / S + 1e-3
    z0[4 * nbld + nbus:] = np.maximum(0.0, v0 - v_max) / S + 1e-3
    res = minimize(obj, z0, jac=jac, hess=hess, method="trust-constr", bounds=Bounds(lo, np.full(nv, np.inf)),
                   constraints=[LinearConstraint(A, lb, np.full(2 * nbus, np.inf))],
                   options={"maxiter": 3000, "gtol": 1e-10, "xtol": 1e-14, "barrier_tol": 1e-12})
    return res.x[:4 * nbld].reshape(nbld, 4) * S, res


# ---------------------------------------------------------------------------------------------------------------------
# The safety layer against the full affine map V = A [P_1, Q_1, ..., P_nb, Q_nb] + c (fp_safety_project_affine).
#
# V depends on the actions only through z = (u_1..u_na, g_1..g_na), u_k = -Pd x_k + c_k - d_k at building k's bus:
# V(z) = V(z0) + B (z - z0) with B[:, k] = A[:, 2 b_k], B[:, na + k] = A[:, 2 b_k + 1].  For a given u_k the best
# (x, c, d) is the projection of safety_ref.project_closed_form: y(r) = max(y0 + (r / 2) a, 0), a = (-Pd, 1, -1), with r the
# multiplier of a . y = u; so phi_k(u) = min ||y - y0||^2 is C^1, convex, piecewise quadratic with phi_k'(u) = r and
# phi_k''(u) = 1 / s, s = du/dr = sum of a_i^2 / 2 over the variables not clamped at zero (<= 3 breakpoints in r).
# What is left is the 2 na-variable convex problem
#     min_z  sum_k phi_k(u_k) + (g_k - g0_k)^2 + w sum_n h(V_n(z)),   h(v) = max(0, v_min - v) + max(0, v - v_max),
# solved by a primal active-set method: every bus is inside (I), below (L, cost -w V), above (U, cost +w V) or held at a
# limit (working set W, multiplier lam_n); every building sits on one quadratic piece of phi_k.  One iteration takes the
# Newton step of the current piece model subject to V_W = limits (a |W| x |W| SPD solve, |W| <= 2 na: the rows of W stay
# independent because a bus only joins along a direction that keeps the others fixed and moves it; once |W| = 2 na the
# step only corrects rounding and no bus joins) and walks along it, up to the Newton point, through the kinks (a bus
# reaching a limit raises the directional derivative by w |dV_n|) and the buildings' breakpoints (the curvature changes);
# where the derivative turns non-negative on a kink, that bus joins W.  After a full Newton step that crossed nothing
# the multipliers are checked: a bus held at v_min needs lam in [0, w], at v_max lam in [-w, 0]; the worst violator
# leaves W (lam < 0 at v_min: inside; lam > w: below; likewise at v_max), else the point is optimal.
# ---------------------------------------------------------------------------------------------------------------------
AFFINE_MAX_ITER = 64          # iteration cap of fp_safety_project_affine (status -1 when reached)
AFFINE_DV_TOL = 1e-12         # a bus blocks a step only if the full step moves it towards the limit by more than this
AFFINE_LAM_TOL = 1e-9         # relative (to w) tolerance of the multiplier check
ST_IN, ST_LO, ST_HI, ST_AT_MIN, ST_AT_MAX = 0, 1, 2, 3, 4


def affine_prediction(y0, Pd, Qd, agent_bus, A, c):
    """V(y0) = A [P_1, Q_1, ...] + c with the proposal applied at the buildings' buses (Pd, Qd [nb] bus order, slack 0)."""
    P = np.array(Pd, dtype=np.float64); Q = np.array(Qd, dtype=np.float64)
    for k, n in enumerate(agent_bus):
        P[n] = Pd[n] * (1.0 - y0[k, 0]) + y0[k, 1] - y0[k, 2]
        Q[n] = Qd[n] + y0[k, 3]
    x = np.empty(2 * len(P)); x[0::2] = P; x[1::2] = Q
    return np.asarray(A, dtype=np.float64) @ x + np.asarray(c, dtype=np.float64)


def affine_cost(y, y0, Pd, Qd, agent_bus, A, c, v_min, v_max, w=W_SLACK):
    V = affine_prediction(y, Pd, Qd, agent_bus, A, c)
    return float(((y - y0) ** 2).sum()) + w * float((np.maximum(0.0, v_min - V) + np.maximum(0.0, V - v_max)).sum())


def _piece_bounds(brk, j):
    lo = -np.inf if j == 0 else brk[j - 1]
    hi = np.inf if j == 3 else brk[j]
    return lo, hi


def _piece_slope(a, t, lo, hi):
    """du/dr on the piece [lo, hi] of r: variables with a_i > 0 are free above their breakpoint, a_i < 0 below."""
    s = 0.0
    for i in range(3):
        if (a[i] > 0.0 and lo >= t[i]) or (a[i] < 0.0 and hi <= t[i]):
            s += a[i] * a[i] * 0.5
    return s


def project_affine(y0, Pd, Qd, agent_bus, A, c, v_min, v_max, w=W_SLACK, max_iter=AFFINE_MAX_ITER):
    """One env: y0 [na, 4] proposed (x, c, d, g); Pd, Qd [nb] the current demands in bus order (0 at the slack bus);
    agent_bus [na] bus positions of the buildings; A [nb, 2 nb], c [nb].  Returns (y* [na, 4], slack [nb], status):
    status = iterations (0: every bus already inside, y* = y0) or -1 if the cap was reached.  A non-finite V(y0) (a NaN
    in the proposal: parse_actions keeps a NaN action as numpy.clip does) leaves the env unprojected: y* = y0 with its
    NaN, slack 0 on every bus, status 0."""
    y0 = np.asarray(y0, dtype=np.float64); agent_bus = np.asarray(agent_bus, dtype=np.int64)
    A = np.asarray(A, dtype=np.float64)
    na, nb = len(agent_bus), len(Pd)
    V0 = affine_prediction(y0, Pd, Qd, agent_bus, A, c)
    if not np.isfinite(V0).all() or ((V0 >= v_min) & (V0 <= v_max)).all():
        return y0.copy(), np.zeros(nb), 0
    B = np.concatenate([A[:, 2 * agent_bus], A[:, 2 * agent_bus + 1]], axis=1)          # [nb, 2 na]
    a = np.stack([-np.asarray(Pd, dtype=np.float64)[agent_bus], np.ones(na), -np.ones(na)], axis=1)
    t = np.full((na, 3), np.inf)                      # breakpoint of each bounded variable (inf: a_i = 0, never clamps)
    nz = a != 0.0
    t[nz] = -2.0 * y0[:, :3][nz] / a[nz]
    brk = np.sort(t, axis=1)
    piece = (brk <= 0.0).sum(axis=1)                  # the piece [lo, hi) holding r = 0
    r = np.zeros(na)
    dz = np.zeros(2 * na)
    st = np.where(V0 < v_min, ST_LO, np.where(V0 > v_max, ST_HI, ST_IN))
    work = []
    released, released_lim = -1, 0.0
    status = -1
    for it in range(max_iter):
        s = np.array([_piece_slope(a[k], t[k], *_piece_bounds(brk[k], piece[k])) for k in range(na)])
        hinv = np.concatenate([s, np.full(na, 0.5)])
        coef = np.where(st == ST_LO, w, np.where(st == ST_HI, -w, 0.0))
        grad = np.concatenate([r, 2.0 * dz[na:]]) - B.T @ coef
        V = V0 + B @ dz
        lam = np.zeros(0)
        if work:
            Bw = B[work]
            M = (Bw * hinv) @ Bw.T
            tgt = np.where(st[work] == ST_AT_MIN, v_min, v_max)
            lam = np.linalg.solve(M, (tgt - V[work]) + Bw @ (hinv * grad))
            p = hinv * (Bw.T @ lam - grad)
        else:
            p = -hinv * grad
        dV = B @ p
        # line search along p up to the Newton point: walk the kinks (a bus reaching a limit: the slope jumps by w |dV_n|) and the
        # buildings' piece breakpoints (the curvature changes) while the directional derivative stays negative
        D = float(grad @ p)
        kappa = float((p * p / hinv).sum())
        cur, crossed, joined = 0.0, False, False
        while kappa > 0.0:
            ev_a, ev = np.inf, None
            if len(work) < 2 * na:                        # W full: the step only corrects rounding, no bus joins
                for n in range(nb):
                    if st[n] >= ST_AT_MIN or abs(dV[n]) <= AFFINE_DV_TOL:
                        continue
                    if dV[n] > 0.0 and st[n] != ST_HI:
                        lim = v_max if st[n] == ST_IN else v_min
                    elif dV[n] < 0.0 and st[n] != ST_LO:
                        lim = v_min if st[n] == ST_IN else v_max
                    else:
                        continue
                    if n == released and lim == released_lim:    # the kink it just left: it moves away from it
                        continue
                    an = max(cur, (lim - V[n]) / dV[n])
                    if an < ev_a:
                        ev_a, ev = an, ("bus", n, lim)
            for k in range(na):
                dr = p[k] / s[k]
                lo, hi = _piece_bounds(brk[k], piece[k])
                if dr > 0.0 and hi < np.inf:
                    ak, side = cur + max(0.0, (hi - r[k]) / dr), 1
                elif dr < 0.0 and lo > -np.inf:
                    ak, side = cur + max(0.0, (lo - r[k]) / dr), -1
                else:
                    continue
                if ak < ev_a:
                    ev_a, ev = ak, ("piece", k, side)
            # the minimum of the current segment's quadratic, at most the Newton point (exact on W's equalities)
            stop = 1.0 if not crossed else min(1.0, cur - D / kappa)
            if ev is None or ev_a >= stop:
                r += (stop - cur) * p[:na] / s
                cur = stop
                break
            D += kappa * (ev_a - cur)
            r += (ev_a - cur) * p[:na] / s
            cur, crossed = ev_a, True
            if ev[0] == "bus":
                n, lim = ev[1], ev[2]
                D += w * abs(dV[n])
                if D >= 0.0:                              # the minimum sits on this kink: the bus joins W
                    st[n] = ST_AT_MIN if lim == v_min else ST_AT_MAX
                    work.append(n)
                    joined = True
                    break
                st[n] = ST_IN if st[n] != ST_IN else (ST_HI if lim == v_max else ST_LO)
            else:
                k = ev[1]
                lo, hi = _piece_bounds(brk[k], piece[k])
                r[k] = hi if ev[2] > 0 else lo
                piece[k] += ev[2]
                s_new = _piece_slope(a[k], t[k], *_piece_bounds(brk[k], piece[k]))
                kappa += p[k] * p[k] * (1.0 / s_new - 1.0 / s[k])
                s[k] = s_new
        dz += cur * p
        if cur > 0.0:
            released = -1
        if crossed or joined:
            continue
        # a full Newton step with nothing crossed: check the multipliers of W
        viol = np.zeros(len(work))
        for i, n in enumerate(work):
            viol[i] = max(-lam[i], lam[i] - w) if st[n] == ST_AT_MIN else max(lam[i], -w - lam[i])
        if len(work) == 0 or viol.max() <= AFFINE_LAM_TOL * w:
            status = it + 1
            break
        i = int(np.argmax(viol))
        n = work.pop(i)
        released, released_lim = n, (v_min if st[n] == ST_AT_MIN else v_max)
        if st[n] == ST_AT_MIN:
            st[n] = ST_IN if lam[i] < 0.0 else ST_LO
        else:
            st[n] = ST_IN if lam[i] > 0.0 else ST_HI
    y = y0.copy()
    y[:, :3] = np.maximum(y0[:, :3] + 0.5 * r[:, None] * a, 0.0)
    y[:, 3] = y0[:, 3] + dz[na:]
    # the prediction at the returned point; buses held at a limit have no slack by construction
    dzf = np.concatenate([(a * (y[:, :3] - y0[:, :3])).sum(axis=1), y[:, 3] - y0[:, 3]])
    V = V0 + B @ dzf
    slack = np.where(st >= ST_AT_MIN, 0.0, np.maximum(0.0, v_min - V) + np.maximum(0.0, V - v_max))
    return y, slack, status
