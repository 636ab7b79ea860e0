"""CPU: the MLP voltage predictor's host side -- the fp64 forward pass of tests/_mlp_ref.py against scikit-learn's own
MLPRegressor pipeline, the extraction of a fitted model (mlp_from_sklearn) and the folding of the MinMax
scalers into its first and last layer (fold_minmax) -- and the C ABI's null-handle answers."""
import warnings

import numpy as np
import pytest

import _mlp_ref as mlp_ref
from oracle import predictor_ref


def _random_mlp(hidden, activation, seed):
    """An MLPRegressor with random weights of the given shape, fitted for one iteration so that sklearn sets it up."""
    from sklearn.exceptions import ConvergenceWarning
    from sklearn.neural_network import MLPRegressor
    rng = np.random.default_rng(seed)
    m = MLPRegressor(hidden_layer_sizes=hidden, activation=activation, max_iter=1, random_state=seed)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", ConvergenceWarning)
        m.fit(rng.uniform(0, 1, (40, 66)), rng.uniform(0, 1, (40, 33)))
    m.coefs_ = [rng.normal(0, 1 / np.sqrt(c.shape[0]), c.shape) for c in m.coefs_]
    m.intercepts_ = [rng.normal(0, 0.1, c.shape) for c in m.intercepts_]
    return m


@pytest.fixture(scope="module")
def fitted():
    """A (100,) relu MLPRegressor fitted on oracle scenarios with the reference's scalers and split."""
    from sklearn.exceptions import ConvergenceWarning
    X, Y = predictor_ref.generate_scenarios(n=300, seed=0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", ConvergenceWarning)
        model, sx, sy = mlp_ref.fit_mlp_pipeline(X, Y, (100,), max_iter=50)
    return model, sx, sy, X


def test_folded_mlp_equals_sklearn_pipeline(fitted):
    from flexgpu.predictor import mlp_from_sklearn
    model, sx, sy, X = fitted
    W, b, act = mlp_from_sklearn(model, sx, sy)
    want = predictor_ref.predict(model, sx, sy, X)
    assert act == "relu"
    assert np.max(np.abs(mlp_ref.mlp_predict(W, b, act, X) - want)) < 1e-12


@pytest.mark.parametrize("hidden,activation", [((64, 64), "tanh"), ((32, 32, 32), "logistic"), ((16,), "identity")])
def test_random_mlps_fold_against_sklearn(hidden, activation):
    from sklearn.preprocessing import MinMaxScaler
    from flexgpu.predictor import mlp_from_sklearn
    rng = np.random.default_rng(len(hidden))
    X = rng.uniform(0.0, 0.3, (200, 66)); Y = rng.uniform(0.9, 1.05, (200, 33))
    sx, sy = MinMaxScaler().fit(X), MinMaxScaler().fit(Y)
    m = _random_mlp(hidden, activation, 3)
    W, b, act = mlp_from_sklearn(m, sx, sy)
    assert act == activation
    assert [w.shape for w in W] == [(h_out, h_in) for h_in, h_out in zip((66,) + hidden, hidden + (33,))]
    assert [c.shape for c in b] == [(h,) for h in hidden + (33,)]
    want = sy.inverse_transform(m.predict(sx.transform(X)))
    assert np.max(np.abs(mlp_ref.mlp_predict(W, b, act, X) - want)) < 1e-12


def test_unfolded_extraction_and_fold_minmax():
    from flexgpu.predictor import fold_minmax, mlp_from_sklearn
    m = _random_mlp((64,), "tanh", 5)
    W, b, act = mlp_from_sklearn(m)
    assert [w.shape for w in W] == [(64, 66), (33, 64)] and act == "tanh"
    assert np.array_equal(W[0], m.coefs_[0].T) and np.array_equal(b[1], m.intercepts_[1])
    rng = np.random.default_rng(0)
    xs, xm = rng.uniform(0.5, 4, 66), rng.uniform(-1, 0, 66)
    ys, ym = rng.uniform(2, 9, 33), rng.uniform(-8, -6, 33)
    Wf, bf = fold_minmax(W, b, xs, xm, ys, ym)
    X = rng.uniform(0, 0.3, (100, 66))
    want = (mlp_ref.mlp_predict(W, b, act, X * xs + xm) - ym) / ys
    assert np.max(np.abs(mlp_ref.mlp_predict(Wf, bf, act, X) - want)) < 1e-12
    assert np.array_equal(W[0], m.coefs_[0].T)                          # the inputs are left as they were
    Wi, bi = fold_minmax(W, b)
    assert all(np.array_equal(p, q) for p, q in zip(Wi + bi, W + b))


def test_non_identity_output_activation_is_rejected():
    from flexgpu.predictor import mlp_from_sklearn
    m = _random_mlp((16,), "relu", 1)
    m.out_activation_ = "logistic"
    with pytest.raises(ValueError, match="output activation"):
        mlp_from_sklearn(m)


def test_null_handle_calls_are_rejected():
    import ctypes as C
    from flexgpu import _lib
    l = _lib.lib()
    widths = (C.c_int32 * 3)(66, 16, 33)
    assert l.fp_predictor_load_mlp(None, 2, widths, None, None, 1, 0.9, 1.1, 1000.0) == -1
    assert l.fp_predict_mlp(None, 0, None, None, None, None, 0, 0, 0, None) == -1
