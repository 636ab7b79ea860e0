"""fp64 reference for the MLP voltage predictor (test infrastructure): the reference's training pipeline with its
regressor swapped for scikit-learn's MLPRegressor, and the fp64 forward pass of the layers that flexgpu loads."""
import numpy as np


def fit_mlp_pipeline(X, Y, hidden, random_state=0, test_size=0.2, split_state=42, **mlp_kw):
    """oracle.predictor_ref.fit_pipeline (train_safety_signal_model.py:33-46: MinMax scalers on X and Y, 80/20 split)
    with MLPRegressor(hidden_layer_sizes=hidden) in place of MultiOutputRegressor(LinearRegression())."""
    from sklearn.model_selection import train_test_split
    from sklearn.neural_network import MLPRegressor
    from sklearn.preprocessing import MinMaxScaler
    sx, sy = MinMaxScaler(), MinMaxScaler()
    Xs, Ys = sx.fit_transform(X), sy.fit_transform(Y)
    Xtr, Xte, Ytr, Yte = train_test_split(Xs, Ys, test_size=test_size, random_state=split_state)
    model = MLPRegressor(hidden_layer_sizes=tuple(hidden), random_state=random_state, **{"max_iter": 2000, **mlp_kw}).fit(Xtr, Ytr)
    return model, sx, sy


def mlp_predict(weights, biases, activation, X):
    """fp64 forward pass of an MLPRegressor's layers (weights [out, in]): act on every hidden layer, identity output."""
    acts = {"identity": lambda z: z, "relu": lambda z: np.maximum(z, 0.0), "tanh": np.tanh,
            "logistic": lambda z: 1.0 / (1.0 + np.exp(-z))}
    h = np.asarray(X, dtype=np.float64)
    for l, (W, b) in enumerate(zip(weights, biases)):
        h = h @ np.asarray(W, dtype=np.float64).T + np.asarray(b, dtype=np.float64)
        if l < len(weights) - 1:
            h = acts[activation](h)
    return h
