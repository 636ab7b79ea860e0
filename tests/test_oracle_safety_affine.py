"""CPU: the active-set projection against the full affine voltage map (oracle/safety_affine_ref.py project_affine, what
k_safety_project_affine implements) against the same QP handed to a generic solver (solve_affine_qp, scipy
trust-constr), against the closed form on a row-sum map, and against random perturbations (first-order optimality)."""
import numpy as np
import pytest

from oracle import safety_affine_ref, safety_ref

BLDS = np.array([4, 9, 14, 19, 24])                                # bus positions of buildings 5, 10, 15, 20, 25
NB = 33


def _proposal(rng):
    y0 = np.stack([rng.uniform(0, 0.5, 5), rng.uniform(0, 0.005, 5), rng.uniform(0, 0.005, 5), rng.uniform(-0.02, 0.02, 5)], axis=1)
    y0[rng.random(5) < 0.5, 1] = 0.0; y0[y0[:, 1] > 0, 2] = 0.0              # never both charging and discharging
    return y0


def _dense_case(rng, kind):
    """Pd, Qd in bus order (0 at the slack bus), a dense map with more load -> lower voltage, and an intercept placed so
    that the proposal is inside, a little low (recoverable), high, hopelessly low, or a mix."""
    Pd = rng.uniform(0.02, 0.4, NB); Qd = rng.uniform(0.01, 0.2, NB); Pd[0] = Qd[0] = 0.0
    A = -rng.uniform(0.0, 0.02, (NB, 2 * NB))                    # the magnitudes of a feeder's sensitivities (p.u.)
    A[:, 2 * BLDS] -= rng.uniform(0.005, 0.06, (NB, 5)); A[:, 2 * BLDS + 1] -= rng.uniform(0.002, 0.04, (NB, 5))
    y0 = _proposal(rng)
    V_free = safety_affine_ref.affine_prediction(y0, Pd, Qd, BLDS, A, np.zeros(NB))
    if kind == "inside":
        c = 1.0 - V_free
    elif kind == "low":
        c = 0.9 - V_free - rng.uniform(0.0, 0.002, NB)
    elif kind == "high":
        c = 1.1 - V_free + rng.uniform(0.0, 0.002, NB)
    elif kind == "hopeless":
        c = 0.9 - V_free - rng.uniform(500.0, 4000.0, NB)
    else:
        c = 1.0 - V_free + rng.uniform(-0.12, 0.12, NB)
    return y0, Pd, Qd, A, c


def _is_building():
    is_b = -np.ones(NB, dtype=int)
    is_b[BLDS] = np.arange(5)
    return is_b


@pytest.mark.parametrize("kind", ["inside", "low", "high", "hopeless", "mixed"])
def test_active_set_matches_the_posed_qp(kind):
    rng = np.random.default_rng({"inside": 11, "low": 12, "high": 13, "hopeless": 14, "mixed": 15}[kind])
    y0, Pd, Qd, A, c = _dense_case(rng, kind)
    got, slack, status = safety_affine_ref.project_affine(y0, Pd, Qd, BLDS, A, c, 0.9, 1.1)
    if kind == "inside":                                             # no solver call: the proposal is returned as is
        assert status == 0 and np.array_equal(got, y0) and not slack.any()
        return
    assert status > 0, status
    want, _ = safety_affine_ref.solve_affine_qp(y0, Pd, Qd, _is_building(), A, c, 0.9, 1.1)    # ~7 s per case
    cost = lambda y: safety_affine_ref.affine_cost(y, y0, Pd, Qd, BLDS, A, c, 0.9, 1.1)
    assert cost(got) <= cost(want) * (1 + 1e-7) + 1e-9, (kind, cost(got), cost(want))
    assert (got[:, :3] >= 0).all()
    scale = max(1.0, float(np.abs(want - y0).max()))
    assert np.max(np.abs(got - want)) < 1e-6 * scale, (kind, np.max(np.abs(got - want)))
    V = safety_affine_ref.affine_prediction(got, Pd, Qd, BLDS, A, c)
    assert np.allclose(slack, np.maximum(0.0, 0.9 - V) + np.maximum(0.0, V - 1.1), rtol=1e-9, atol=1e-12)
    if kind == "hopeless":
        assert (slack > 0).all()


def test_posing_is_the_reference_qp_on_row_sums():
    """posed_qp with the row-sum prediction poses exactly the QP of safety_ref.solve_reference_qp: same solver path,
    same optimum, to the bit."""
    rng = np.random.default_rng(31)
    Pd = rng.uniform(0.02, 0.4, NB); Qd = rng.uniform(0.01, 0.2, NB)
    sP = rng.uniform(-0.9, -0.05, NB); sQ = rng.uniform(-0.6, -0.02, NB)
    y0 = _proposal(rng)
    b = 1.0 - sP * Pd - sQ * Qd + rng.uniform(-0.25, 0.25, NB)
    want, _ = safety_ref.solve_reference_qp(y0, Pd, Qd, _is_building(), sP, sQ, b, 0.9, 1.1)
    got, _ = safety_affine_ref.posed_qp(y0, Pd, Qd, _is_building(), lambda P, Q: sP * P + sQ * Q + b, 0.9, 1.1,
                                        safety_ref.W_SLACK)
    assert np.array_equal(got, want)


def test_row_sum_map_is_the_closed_form():
    """With the reference's 2-banded map (bus n sees only its own P_n, Q_n) the problem separates per building and the
    active-set method must land on project_closed_form's point."""
    rng = np.random.default_rng(21)
    for trial in range(60):
        Pd = rng.uniform(0.02, 0.4, NB); Qd = rng.uniform(0.01, 0.2, NB); Pd[0] = Qd[0] = 0.0
        sP = rng.uniform(-0.9, -0.05, NB); sQ = rng.uniform(-0.6, -0.02, NB)
        y0 = _proposal(rng)
        b = 1.0 - sP * Pd - sQ * Qd + rng.uniform(-0.3, 0.3, NB)
        A = np.zeros((NB, 2 * NB)); A[np.arange(NB), 2 * np.arange(NB)] = sP; A[np.arange(NB), 2 * np.arange(NB) + 1] = sQ
        got, slack, status = safety_affine_ref.project_affine(y0, Pd, Qd, BLDS, A, b, 0.9, 1.1)
        assert status >= 0
        for k, n in enumerate(BLDS):
            want, wslack, _ = safety_ref.project_closed_form(y0[k], Pd[n], Qd[n], sP[n], sQ[n], b[n], 0.9, 1.1)
            assert np.max(np.abs(got[k] - want)) <= 1e-12, (trial, k, got[k], want)
            assert abs(slack[n] - wslack) <= 1e-12, (trial, k, slack[n], wslack)


def test_active_set_kkt_on_random_cases():
    """First-order optimality without any solver: no feasible perturbation lowers the exact-penalty cost."""
    rng = np.random.default_rng(22)
    iters = []
    for trial in range(100):
        y0, Pd, Qd, A, c = _dense_case(rng, rng.choice(["low", "high", "mixed", "hopeless"]))
        y, slack, status = safety_affine_ref.project_affine(y0, Pd, Qd, BLDS, A, c, 0.9, 1.1)
        assert status > 0, (trial, status)
        iters.append(status)
        cost = lambda z: safety_affine_ref.affine_cost(z, y0, Pd, Qd, BLDS, A, c, 0.9, 1.1)
        c0 = cost(y)
        for _ in range(30):
            z = y + rng.normal(0, 1e-4, y.shape) * rng.choice([1.0, 10.0, 100.0])
            z[:, :3] = np.maximum(z[:, :3], 0.0)
            assert cost(z) >= c0 - 1e-12 * max(1.0, c0), trial
    assert max(iters) < safety_affine_ref.AFFINE_MAX_ITER


@pytest.mark.parametrize("kind", ["low", "high", "mixed", "hopeless"])
def test_nan_proposal_is_left_unprojected(kind):
    """A NaN in the proposal (parse_actions keeps a NaN action, as numpy.clip does) makes V(y0) non-finite: the env is
    returned as proposed, NaN included, with no slack and status 0 -- what k_safety_project_affine writes."""
    rng = np.random.default_rng({"low": 41, "high": 42, "mixed": 43, "hopeless": 44}[kind])
    y0, Pd, Qd, A, c = _dense_case(rng, kind)
    assert safety_affine_ref.project_affine(y0, Pd, Qd, BLDS, A, c, 0.9, 1.1)[2] > 0      # finite: it moves
    for k in range(5):
        for i in range(4):
            bad = y0.copy(); bad[k, i] = np.nan
            got, slack, status = safety_affine_ref.project_affine(bad, Pd, Qd, BLDS, A, c, 0.9, 1.1)
            assert status == 0 and np.array_equal(slack, np.zeros(NB))
            assert np.array_equal(got, bad, equal_nan=True) and np.isnan(got[k, i]) and np.isnan(got).sum() == 1
