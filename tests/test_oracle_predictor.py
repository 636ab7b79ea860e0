"""CPU: pins the predictor / replay oracle against scikit-learn's own pipeline (the golden fixture
was produced by sklearn fit + predict, tests/golden/make_golden.py) and the reference's
TransReplayBuffer semantics (utils/replay_buffer.py:3-30)."""
import os

import numpy as np
import pytest

from oracle import predictor_ref, replay_ref
from _golden import load_ref_predictor

GOLD = os.path.join(os.path.dirname(__file__), "golden", "predictor_golden.npz")


def fold(g):
    """The host-side folding flexgpu.predictor.VoltagePredictor.from_linear_model performs."""
    W, b = g["coef"], g["intercept"]
    A = W * g["x_scale"][None, :] / g["y_scale"][:, None]
    c = (W @ g["x_min"] + b - g["y_min"]) / g["y_scale"]
    return A, c


def test_folded_affine_map_equals_sklearn_predict():
    g = np.load(GOLD)
    A, c = fold(g)
    V = predictor_ref.affine_predict(A, c, g["X"])
    assert np.max(np.abs(V - g["V"])) < 1e-12
    assert np.max(np.abs(predictor_ref.slack_penalty(V) - g["penalty"])) < 1e-8
    assert (g["penalty"] == 0.0).sum() >= 5 and g["penalty"].max() > 1000.0             # both regimes are in the fixture
    assert abs(g["V"][:, 0] - 1.0).max() < 1e-12                                     # slack bus: constant column


def test_pipeline_reproduces_itself():
    X, Y = predictor_ref.generate_scenarios(60, seed=0)
    m, sx, sy = predictor_ref.fit_pipeline(X, Y)
    P = predictor_ref.predict(m, sx, sy, X)
    assert X.shape == (60, 66) and Y.shape == (60, 33) and np.max(np.abs(P - Y)) < 5e-3
    assert np.all(X[:, 0] == 0) and np.all(X[:, 1] == 0)                             # slack bus has no load
    assert np.allclose(X[:, 2::2].mean(0) / X[:, 2::2].mean(0), 1.0)


def test_rowsum_quirk_form_differs_from_the_proper_map():
    g = np.load(GOLD)
    V = predictor_ref.rowsum_predict(g["coef"], g["intercept"], g["X"])
    assert np.array_equal(V, g["V_rowsum"]) and np.max(np.abs(V - g["V"])) > 1e-3      # it is a different model


def test_replay_fifo_and_contiguous_window():
    buf = replay_ref.RefTransReplayBuffer(5)
    for i in range(8):
        buf.add_experience({"x": np.array([i], dtype=np.float32)})
    assert len(buf) == 5 and [int(t["x"][0]) for t in buf.buffer] == [3, 4, 5, 6, 7]    # oldest popped (:23-27)
    rng = np.random.RandomState(0)
    for _ in range(20):
        batch, start = buf.get_batch(3, rng)
        assert 0 <= start <= 2 and [int(t["x"][0]) for t in batch] == [3 + start, 4 + start, 5 + start]   # consecutive (:17-20)
    buf.clear()
    assert len(buf) == 0
    with pytest.raises(ValueError):
        buf.get_batch(1, rng)


# ---------------------------------------------------------------------------------------------------
# PIN on the reference's own scripts: tests/golden/ref_predictor.npz holds what safety_signal/data_generation.py
# and train_safety_signal_model.py (executed unchanged, file I/O intercepted) produced -- the 1000 scenarios, the
# fitted regressor, the scalers the script forgets to save, and its own predictions.
# The scenarios X are redrawn by tests/_golden.py and checked against the SHA-256 of the reference's bytes.


def test_oracle_scenarios_equal_the_reference_script():
    g = load_ref_predictor()
    X, Y = predictor_ref.generate_scenarios(40, seed=2024)         # same stream: 33 P draws then 33 Q draws per scenario
    assert np.array_equal(X, g["X"][:40])
    assert np.max(np.abs(Y - g["Y"][:40])) < 1e-10                 # sweep vs Newton behind the reference's model


def test_oracle_fit_equals_the_reference_fit():
    g = load_ref_predictor()
    m, sx, sy = predictor_ref.fit_pipeline(g["X"], g["Y"])
    coef = np.array([e.coef_ for e in m.estimators_])
    # the slack-bus columns of X and Y are constant (scale 1, all-zero scaled column): their coefficients are
    # arbitrary minimum-norm values, everything else is the unique least-squares solution
    assert np.allclose(sx.scale_, g["x_scale"], rtol=0, atol=0) and np.allclose(sy.min_, g["y_min"], rtol=0, atol=0)
    V = predictor_ref.predict(m, sx, sy, g["X"])
    assert np.max(np.abs(V - g["V_pred"])) < 1e-9
    assert np.max(np.abs(coef - g["coef"])) < 1e-6


def test_folded_affine_map_equals_the_reference_predictions():
    """The host-side folding (VoltagePredictor.from_linear_model) applied to the reference's regressor and scalers
    reproduces (i) sklearn's predictions in p.u. for all 1000 scenarios and (ii) the scaled predictions the
    reference's script itself computed on its test split (train_safety_signal_model.py:76)."""
    g = load_ref_predictor()
    A, c = fold(g)
    V = predictor_ref.affine_predict(A, c, g["X"])
    assert np.max(np.abs(V - g["V_pred"])) < 1e-12
    Xte = (g["X_test_scaled"] - g["x_min"]) / g["x_scale"]          # un-scale the script's test inputs
    Vte = predictor_ref.affine_predict(A, c, Xte)
    assert np.max(np.abs(Vte * g["y_scale"] + g["y_min"] - g["Y_pred_scaled"])) < 1e-9
    assert float(g["r2"][0]) > 0.999 and np.max(np.abs(V - g["Y"])) < 5e-3


def test_replay_restatement_equals_the_reference_class():
    """oracle/replay_ref.py against utils/replay_buffer.py::TransReplayBuffer itself (imported by the generator):
    same adds, same numpy seed -> same window starts and the same transitions in every batch."""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_replay.npz"))
    buf = replay_ref.RefTransReplayBuffer(int(g["size"][0]))
    np.random.seed(int(g["seed"][0]))
    n_added, k = 0, 0
    for n_target, batch in g["events"]:
        while n_added < n_target:
            buf.add_experience(g["rows"][n_added]); n_added += 1
        got, start = buf.get_batch(int(batch))
        assert start == g["starts"][k] and [int(t[0]) for t in got] == list(g["ids"][k][:batch])
        k += 1
    assert [int(t[0]) for t in buf.buffer] == list(g["final_ids"])
