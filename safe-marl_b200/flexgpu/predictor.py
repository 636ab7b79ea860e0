"""Safety-signal voltage predictor (tcgen05) and the device-resident replay ring.

VoltagePredictor   batched `model.predict` of the reference's regressor
                   (safety_signal/train_safety_signal_model.py:33-46,73: MinMaxScaler on X and Y +
                   MultiOutputRegressor(LinearRegression), 66 -> 33) plus the safety layer's slack
                   penalty (madrl/models/safemaddpg.py:205-229), through fp_predict.
MLPVoltagePredictor the same for a scikit-learn MLPRegressor swapped in for the regressor (1..3 hidden
                   layers of width <= 128), through fp_predict_mlp; mlp_from_sklearn / fold_minmax turn the
                   fitted model and its scalers into the raw-input layers it loads.
DeviceReplayBuffer TransReplayBuffer (utils/replay_buffer.py:3-30) as a struct-of-arrays fp32 ring
                   on the device, through fp_replay_*.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


class DeviceReplayBuffer:
    """FIFO of `size` transitions; every field is a [size, width] fp32 ring on the device."""

    def __init__(self, size, fields, device="cuda:0"):
        self.size = int(size)                                              # :5
        self.fields = dict(fields)
        self.names = list(self.fields)
        self.device = torch.device(device)
        if self.device.type != "cuda" or not torch.cuda.is_available():
            raise _lib.FlexGpuError("DeviceReplayBuffer needs a CUDA device; there is no CPU fallback")
        self._lib = _lib.lib()
        self._r = C.c_void_p()
        widths = (C.c_int32 * len(self.names))(*[int(self.fields[k]) for k in self.names])
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", idx)
        _lib.check(self._lib.fp_replay_create(self.size, len(self.names), widths, idx, C.byref(self._r)), None, "fp_replay_create",
                   self._lib.fp_replay_last_error)

    def _check(self, rc, what):
        _lib.check(rc, self._r, what, self._lib.fp_replay_last_error)

    def close(self):
        if getattr(self, "_r", None) is not None and self._r.value:
            self._lib.fp_replay_destroy(self._r)
            self._r = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self):
        return int(self._lib.fp_replay_len(self._r))

    def clear(self):                                                       # :29-30
        self._check(self._lib.fp_replay_clear(self._r), "fp_replay_clear")

    def reserve(self, n):
        """Make room for n new rows (oldest rows are dropped when full) -> ring position."""
        pos = C.c_int64()
        self._check(self._lib.fp_replay_reserve(self._r, int(n), C.byref(pos)), "fp_replay_reserve")
        return pos.value

    def write(self, name, pos, rows):
        f = self.names.index(name)
        rows = rows.to(device=self.device, dtype=torch.float32).contiguous().view(-1, self.fields[name])
        self._check(self._lib.fp_replay_write(self._r, f, int(pos), rows.shape[0], _ptr(rows), _lib.stream(self.device)), "fp_replay_write")

    def add_experience(self, trans):                                       # :23-27, n rows at once
        n = next(iter(trans.values())).shape[0]
        if n > self.size:                      # more rows than the FIFO holds: all but the last `size` are popped again
            trans = {k: v[n - self.size:] for k, v in trans.items()}
            n = self.size
        pos = self.reserve(n)
        for k, v in trans.items():
            self.write(k, pos, v)
        return pos

    def get_batch(self, batch_size, start=None):                           # :14-21
        sample_range = len(self) - batch_size + 1
        if sample_range < 1:
            raise ValueError("batch larger than the buffer")
        if start is None:
            start = int(np.random.choice(sample_range, 1, replace=False)[0])   # the reference's draw (:18)
        out = {k: torch.empty(batch_size, w, dtype=torch.float32, device=self.device) for k, w in self.fields.items()}
        ptrs = (C.c_void_p * len(self.names))(*[out[k].data_ptr() for k in self.names])
        self._check(self._lib.fp_replay_sample(self._r, int(start), int(batch_size), ptrs, _lib.stream(self.device)), "fp_replay_sample")
        return out


class VoltagePredictor:
    """Vhat = A x + c on raw interleaved inputs x = [P1, Q1, ..., P33, Q33] (data_generation.py:48-50)."""

    def __init__(self, env, A, c, v_min=None, v_max=None, slack_weight=1000.0):
        self.env = env
        self.A = np.ascontiguousarray(A, dtype=np.float64)
        self.c = np.ascontiguousarray(c, dtype=np.float64)
        self.n_out, self.n_in = self.A.shape
        self.v_min = float(env.args_dict["v_min"] if v_min is None else v_min)
        self.v_max = float(env.args_dict["v_max"] if v_max is None else v_max)
        self.slack_weight = float(slack_weight)                            # safemaddpg.py:229 (1000)
        self._load()

    def _load(self):
        """The handle holds ONE model (fp_predictor_load); several VoltagePredictor objects may share a
        handle, so each (re)loads its weights when it is not the one currently resident."""
        env = self.env
        env._check(env._lib.fp_predictor_load(env._h, self.n_in, self.n_out, self.A.ctypes.data_as(C.c_void_p),
                                              self.c.ctypes.data_as(C.c_void_p), self.v_min, self.v_max,
                                              self.slack_weight), "fp_predictor_load")
        env._resident_predictor = self

    @classmethod
    def from_linear_model(cls, env, coef, intercept, x_scale=None, x_min=None, y_scale=None, y_min=None, **kw):
        """coef [33, 66], intercept [33] of the fitted regressor; x_scale/x_min and y_scale/y_min are
        sklearn MinMaxScaler.scale_/min_ of the X and Y scalers (train_safety_signal_model.py:34-37).
        The scalers are folded into one affine map in fp64."""
        W = np.asarray(coef, dtype=np.float64); b = np.asarray(intercept, dtype=np.float64)
        sx = np.ones(W.shape[1]) if x_scale is None else np.asarray(x_scale, dtype=np.float64)
        mx = np.zeros(W.shape[1]) if x_min is None else np.asarray(x_min, dtype=np.float64)
        sy = np.ones(W.shape[0]) if y_scale is None else np.asarray(y_scale, dtype=np.float64)
        my = np.zeros(W.shape[0]) if y_min is None else np.asarray(y_min, dtype=np.float64)
        A = W * sx[None, :] / sy[:, None]
        c = (W @ mx + b - my) / sy
        return cls(env, A, c, **kw)

    @classmethod
    def from_sklearn(cls, env, model, scaler_x=None, scaler_y=None, **kw):
        coef = np.array([e.coef_ for e in model.estimators_]) if hasattr(model, "estimators_") else model.coef_
        icpt = np.array([e.intercept_ for e in model.estimators_]) if hasattr(model, "estimators_") else model.intercept_
        return cls.from_linear_model(env, coef, icpt,
                                     None if scaler_x is None else scaler_x.scale_, None if scaler_x is None else scaler_x.min_,
                                     None if scaler_y is None else scaler_y.scale_, None if scaler_y is None else scaler_y.min_, **kw)

    @classmethod
    def from_safemaddpg_rowsum(cls, env, coef, intercept, **kw):
        """The form the reference's safety layer actually evaluates (safemaddpg.py:182-184,266,272):
        V_i = (sum_j coef[i, :33]) P_i + (sum_j coef[i, 33:]) Q_i + b_i -- a 2-banded affine map."""
        W = np.asarray(coef, dtype=np.float64)
        n = W.shape[0]
        A = np.zeros((n, 2 * n))
        A[np.arange(n), 2 * np.arange(n)] = W[:, :n].sum(axis=1)
        A[np.arange(n), 2 * np.arange(n) + 1] = W[:, n:].sum(axis=1)
        return cls(env, A, np.asarray(intercept, dtype=np.float64), **kw)

    def predict(self, X, want_vhat=True, want_penalty=True, sink=None, vhat_field="v_pred",
                penalty_field="safety_penalty", pos=None):
        """X [n, 66] fp32 on the device -> (Vhat [n, 33] fp32, penalty [n] fp64).  With `sink`
        (a DeviceReplayBuffer) the kernel's epilogue also writes both into the ring rows `pos`..
        (reserved here if pos is None)."""
        env = self.env
        if getattr(env, "_resident_predictor", None) is not self:
            self._load()
        X = X.to(device=env.device, dtype=torch.float32).contiguous()
        n = X.shape[0]
        if X.shape[1] != self.n_in:
            raise ValueError("X must be [n, 66]")
        vhat = torch.empty(n, self.n_out, dtype=torch.float32, device=env.device) if want_vhat else None
        pen = torch.empty(n, dtype=torch.float64, device=env.device) if want_penalty else None
        r, fv, fp_ = None, -1, -1
        if sink is not None:
            r = sink._r
            fv = sink.names.index(vhat_field) if vhat_field in sink.names else -1
            fp_ = sink.names.index(penalty_field) if penalty_field in sink.names else -1
            if pos is None:
                pos = sink.reserve(n)
        env._check(env._lib.fp_predict(env._h, n, _ptr(X), _ptr(vhat), _ptr(pen), r, fv, fp_, int(pos or 0), _lib.stream(env.device)),
                   "fp_predict")
        return vhat, pen


def mlp_from_sklearn(model, scaler_x=None, scaler_y=None):
    """A fitted MLPRegressor -> (weights [out, in] per layer, biases per layer, activation), fp64, with the MinMax
    scalers (if given) folded into the first and last layer so that the layers act on raw inputs in p.u."""
    if getattr(model, "out_activation_", "identity") != "identity":
        raise ValueError(f"MLPRegressor output activation {model.out_activation_!r}: only 'identity' is supported")
    if model.activation not in _lib.ACTIVATIONS:
        raise ValueError(f"unknown activation {model.activation!r}")
    W = [np.asarray(c, dtype=np.float64).T.copy() for c in model.coefs_]          # sklearn holds [in, out]
    b = [np.asarray(c, dtype=np.float64).copy() for c in model.intercepts_]
    if scaler_x is not None or scaler_y is not None:
        W, b = fold_minmax(W, b, None if scaler_x is None else scaler_x.scale_, None if scaler_x is None else scaler_x.min_,
                           None if scaler_y is None else scaler_y.scale_, None if scaler_y is None else scaler_y.min_)
    return W, b, model.activation

def fold_minmax(weights, biases, x_scale=None, x_min=None, y_scale=None, y_min=None):
    """Folds x_s = x * x_scale + x_min into layer 1 and y = (y_s - y_min) / y_scale into the last layer (sklearn
    MinMaxScaler.scale_ / min_, train_safety_signal_model.py:34-37), in fp64, as from_linear_model does for the
    affine map.  Returns new lists; the inputs are not changed."""
    W = [np.asarray(w, dtype=np.float64) for w in weights]
    b = [np.asarray(c, dtype=np.float64) for c in biases]
    if x_scale is not None:
        sx = np.asarray(x_scale, dtype=np.float64)
        mx = np.zeros_like(sx) if x_min is None else np.asarray(x_min, dtype=np.float64)
        W[0], b[0] = W[0] * sx[None, :], W[0] @ mx + b[0]
    if y_scale is not None:
        sy = np.asarray(y_scale, dtype=np.float64)
        my = np.zeros_like(sy) if y_min is None else np.asarray(y_min, dtype=np.float64)
        W[-1], b[-1] = W[-1] / sy[:, None], (b[-1] - my) / sy
    return W, b


class MLPVoltagePredictor:
    """Vhat = MLP(x) on raw interleaved inputs x = [P1, Q1, ..., P33, Q33]: hidden layers act(W h + b) with one
    activation (identity, relu, tanh, logistic), identity output layer; weights [out, in] per layer.  predict() has
    VoltagePredictor.predict's signature and returns, so either can serve a caller."""

    def __init__(self, env, weights, biases, activation="relu", v_min=None, v_max=None, slack_weight=1000.0):
        self.env = env
        self.weights = [np.ascontiguousarray(w, dtype=np.float64) for w in weights]
        self.biases = [np.ascontiguousarray(c, dtype=np.float64).reshape(-1) for c in biases]
        if len(self.weights) != len(self.biases):
            raise ValueError("one bias vector per weight matrix")
        if activation not in _lib.ACTIVATIONS:
            raise ValueError(f"unknown activation {activation!r} (one of {sorted(_lib.ACTIVATIONS)})")
        self.activation = activation
        self.widths = [self.weights[0].shape[1]] + [w.shape[0] for w in self.weights]
        for l, w in enumerate(self.weights):
            if w.shape != (self.widths[l + 1], self.widths[l]) or self.biases[l].shape != (self.widths[l + 1],):
                raise ValueError(f"layer {l}: weights [out, in] and biases [out] do not chain")
        self.n_in, self.n_out = self.widths[0], self.widths[-1]
        self.v_min = float(env.args_dict["v_min"] if v_min is None else v_min)
        self.v_max = float(env.args_dict["v_max"] if v_max is None else v_max)
        self.slack_weight = float(slack_weight)
        self._load()

    def _load(self):
        """The handle's MLP slot holds ONE model (fp_predictor_load_mlp), separate from the affine model of
        VoltagePredictor; each MLPVoltagePredictor reloads its weights when it is not the resident one."""
        env = self.env
        widths = (C.c_int32 * len(self.widths))(*self.widths)
        W = np.concatenate([w.reshape(-1) for w in self.weights])
        b = np.concatenate(self.biases)
        env._check(env._lib.fp_predictor_load_mlp(env._h, len(self.weights), widths, W.ctypes.data_as(C.c_void_p),
                                                  b.ctypes.data_as(C.c_void_p), _lib.ACTIVATIONS[self.activation],
                                                  self.v_min, self.v_max, self.slack_weight), "fp_predictor_load_mlp")
        env._resident_mlp = self

    @classmethod
    def from_sklearn(cls, env, model, scaler_x=None, scaler_y=None, **kw):
        W, b, act = mlp_from_sklearn(model, scaler_x, scaler_y)
        return cls(env, W, b, activation=act, **kw)

    def predict(self, X, want_vhat=True, want_penalty=True, sink=None, vhat_field="v_pred",
                penalty_field="safety_penalty", pos=None):
        """X [n, 66] fp32 on the device -> (Vhat [n, 33] fp32, penalty [n] fp64), as VoltagePredictor.predict."""
        env = self.env
        if getattr(env, "_resident_mlp", None) is not self:
            self._load()
        X = X.to(device=env.device, dtype=torch.float32).contiguous()
        n = X.shape[0]
        if X.dim() != 2 or X.shape[1] != self.n_in:
            raise ValueError("X must be [n, 66]")
        vhat = torch.empty(n, self.n_out, dtype=torch.float32, device=env.device) if want_vhat else None
        pen = torch.empty(n, dtype=torch.float64, device=env.device) if want_penalty else None
        r, fv, fp_ = None, -1, -1
        if sink is not None:
            r = sink._r
            fv = sink.names.index(vhat_field) if vhat_field in sink.names else -1
            fp_ = sink.names.index(penalty_field) if penalty_field in sink.names else -1
            if pos is None:
                pos = sink.reserve(n)
        env._check(env._lib.fp_predict_mlp(env._h, n, _ptr(X), _ptr(vhat), _ptr(pen), r, fv, fp_, int(pos or 0),
                                           _lib.stream(env.device)), "fp_predict_mlp")
        return vhat, pen


def smoke(env, device):
    """Tiny predictor + replay invocation for __graft_entry__.smoke(): Vhat = identity-ish map."""
    rng = np.random.default_rng(0)
    A = rng.normal(0, 0.05, (33, 66)); c = np.full(33, 1.0)
    pred = VoltagePredictor(env, A, c)
    buf = DeviceReplayBuffer(1000, {"v_pred": 33, "safety_penalty": 1}, device=device)
    X = torch.from_numpy(rng.uniform(-1, 1, (300, 66)).astype(np.float32)).to(device)
    vhat, pen = pred.predict(X, sink=buf)
    want = X.double().cpu().numpy() @ A.T + c
    err = float(np.max(np.abs(vhat.cpu().numpy() - want)))
    assert err < 2e-6, f"predictor mismatch {err}"
    got = buf.get_batch(300, start=0)
    assert torch.equal(got["v_pred"], vhat) and len(buf) == 300
    buf.close()
    return err
