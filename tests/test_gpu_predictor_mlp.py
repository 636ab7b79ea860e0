"""GPU parity: the tcgen05 MLP voltage predictor + safety penalty (fp_predictor_load_mlp / fp_predict_mlp).

Error model, row by row against an fp64 forward pass on the same fp32 X.  It extends the affine
kernel's 3xTF32 bound (2^-20 (|A||x| + |c|)) layer by layer, with the fp32 activation on the CUDA cores:
    e_0 = 0
    ez_l = |W_l| e_{l-1} + 2^-20 (|W_l| |h_{l-1}| + |b_l|)
    e_l  = L_act ez_l + 4 ulp_fp32(|h_l|)          L_act = 1 (identity, relu, tanh), 1/4 (logistic)
The penalty is the fp64 formula on the returned Vhat (exact arithmetic); ring contents are compared bit for bit
with the dense output."""
import ctypes as C
import warnings

import numpy as np
import pytest
import torch

import _mlp_ref as mlp_ref
from oracle import predictor_ref, replay_ref

pytestmark = pytest.mark.gpu
SHAPES = [(16,), (64,), (100,), (128,), (64, 64), (32, 32, 32)]
ACTS = ["identity", "relu", "tanh", "logistic"]
_ACT_T = {"identity": lambda z: z, "relu": torch.relu, "tanh": torch.tanh, "logistic": torch.sigmoid}


def forward_and_bound(W, b, act, X):
    """fp64 forward pass and the per-element error bound above; W, b lists of arrays, X [n, 66] (torch, any device)."""
    h = X.double()
    e = torch.zeros_like(h)
    for l, (w, c) in enumerate(zip(W, b)):
        w = torch.as_tensor(w, dtype=torch.float64, device=h.device); c = torch.as_tensor(c, dtype=torch.float64, device=h.device)
        z = h @ w.T + c
        ez = e @ w.abs().T + 2.0 ** -20 * (h.abs() @ w.abs().T + c.abs())
        hidden = l < len(W) - 1
        h = _ACT_T[act](z) if hidden else z
        lip = 0.25 if (hidden and act == "logistic") else 1.0
        ulp = torch.from_numpy(np.spacing(h.abs().float().cpu().numpy()).astype(np.float64)).to(h.device)
        e = lip * ez + 4.0 * ulp
    return h, e


def random_mlp(hidden, seed):
    rng = np.random.default_rng(seed)
    widths = (66,) + tuple(hidden) + (33,)
    W = [rng.normal(0, 1.0 / np.sqrt(i), (o, i)) for i, o in zip(widths[:-1], widths[1:])]
    b = [rng.normal(0, 0.1, o) for o in widths[1:]]
    b[-1] = b[-1] + 1.0
    return W, b


def pen_ref(v, p):
    vd = v.double()
    return p.slack_weight * (torch.clamp(p.v_min - vd, min=0) + torch.clamp(vd - p.v_max, min=0)).sum(dim=1)


@pytest.fixture(scope="module")
def env(cuda, profiles):
    from flexgpu import BatchedFlexProvisionEnv
    e = BatchedFlexProvisionEnv(None, n_envs=8, device=cuda, profiles=profiles)
    yield e
    e.close()


@pytest.fixture(scope="module")
def fitted():
    """A (100,) relu MLPRegressor on 1000 oracle scenarios, the reference's MinMax scalers and split."""
    X, Y = predictor_ref.generate_scenarios(n=1000, seed=0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model, sx, sy = mlp_ref.fit_mlp_pipeline(X, Y, (100,), random_state=0)
    return model, sx, sy, X


@pytest.fixture(scope="module")
def mlp(env, fitted):
    from flexgpu.predictor import MLPVoltagePredictor
    model, sx, sy, _ = fitted
    return MLPVoltagePredictor.from_sklearn(env, model, sx, sy)


def scenario_inputs(n, seed, device, hi=1.3):
    from flexgpu import DEFAULT_ENV_ARGS, Network, create_network
    net = Network(create_network(DEFAULT_ENV_ARGS))
    base = torch.from_numpy(np.stack([net.base_p, net.base_q], axis=1).reshape(-1)).to(device)
    g = torch.Generator(device=device).manual_seed(seed)
    return (base[None, :] * (0.7 + hi * torch.rand(n, 66, device=device, dtype=torch.float64, generator=g))).float().contiguous()


def test_fitted_relu_mlp_against_sklearn(mlp, fitted, cuda):
    model, sx, sy, X = fitted
    X32 = X.astype(np.float32)
    vhat, pen = mlp.predict(torch.from_numpy(X32).to(cuda))
    V = vhat.cpu().numpy().astype(np.float64)
    want = predictor_ref.predict(model, sx, sy, X32.astype(np.float64))
    _, bound = forward_and_bound(mlp.weights, mlp.biases, "relu", torch.from_numpy(X32))
    assert np.all(np.abs(V - want) <= bound.numpy())
    assert np.max(np.abs(V - want)) < 1e-6
    assert np.allclose(pen.cpu().numpy(), predictor_ref.slack_penalty(V), rtol=1e-12, atol=1e-9)
    v2, p2 = mlp.predict(torch.from_numpy(2 * X32).to(cuda))                  # 2x load: the limits are left somewhere
    want2 = predictor_ref.predict(model, sx, sy, 2 * X32.astype(np.float64))
    _, bound2 = forward_and_bound(mlp.weights, mlp.biases, "relu", torch.from_numpy(2 * X32))
    assert np.all(np.abs(v2.cpu().numpy() - want2) <= bound2.numpy())
    assert int((p2 > 0).sum()) > 0
    assert np.allclose(p2.cpu().numpy(), predictor_ref.slack_penalty(v2.cpu().numpy().astype(np.float64)), rtol=1e-12, atol=1e-9)


@pytest.mark.parametrize("act", ACTS)
@pytest.mark.parametrize("hidden", SHAPES)
def test_shapes_and_activations_every_row_within_bound(env, cuda, hidden, act):
    """Odd sizes take the non-TMA tail path; every row of every launch is inside the layer-by-layer bound."""
    from flexgpu.predictor import MLPVoltagePredictor
    W, b = random_mlp(hidden, len(hidden) * 10 + ACTS.index(act))
    p = MLPVoltagePredictor(env, W, b, activation=act)
    rng = np.random.default_rng(7)
    for n in (1, 2, 127, 128, 129, 1000, 4097):
        X = rng.uniform(-1, 1, (n, 66)).astype(np.float32)
        vhat, pen = p.predict(torch.from_numpy(X).to(cuda))
        want, bound = forward_and_bound(W, b, act, torch.from_numpy(X))
        err = np.abs(vhat.cpu().numpy().astype(np.float64) - want.numpy())
        assert vhat.shape == (n, 33) and np.all(err <= bound.numpy()), (n, float((err / bound.numpy()).max()))
        assert np.allclose(pen.cpu().numpy(), pen_ref(vhat, p).cpu().numpy(), rtol=1e-12, atol=1e-9)


def test_identity_mlp_matches_the_affine_kernel(env, cuda):
    from flexgpu.predictor import MLPVoltagePredictor, VoltagePredictor
    W, b = random_mlp((64,), 11)
    A, c = W[1] @ W[0], W[1] @ b[0] + b[1]
    pm = MLPVoltagePredictor(env, W, b, activation="identity")
    pa = VoltagePredictor(env, A, c)
    X = np.random.default_rng(3).uniform(-1, 1, (1000, 66)).astype(np.float32)
    Xd = torch.from_numpy(X).to(cuda)
    vm, _ = pm.predict(Xd)
    va, _ = pa.predict(Xd)
    _, bm = forward_and_bound(W, b, "identity", torch.from_numpy(X))
    ba = 2.0 ** -20 * (np.abs(X.astype(np.float64)) @ np.abs(A).T + np.abs(c))
    assert np.all(np.abs(vm.cpu().numpy().astype(np.float64) - va.cpu().numpy()) <= bm.numpy() + ba)


def test_rows_are_independent_and_launches_deterministic(mlp, cuda):
    X = scenario_inputs(1000, 5, cuda, hi=1.3)
    v, p = mlp.predict(X)
    v2, p2 = mlp.predict(X)
    assert torch.equal(v, v2) and torch.equal(p, p2)
    for i, j in ((1, 2), (5, 300), (130, 389), (257, 1000), (999, 1000)):
        vs, ps = mlp.predict(X[i:j].clone())                          # a slice that starts mid-tile, as a new launch
        assert torch.equal(vs, v[i:j]) and torch.equal(ps, p[i:j]), (i, j)
    Xn = X.clone()
    Xn[77, 5] = float("nan")
    vn, pn = mlp.predict(Xn)
    keep = torch.arange(1000, device=cuda) != 77
    assert torch.equal(vn[keep], v[keep]) and torch.equal(pn[keep], p[keep])
    assert bool(torch.isnan(vn[77]).any())


@pytest.mark.parametrize("n", [127, 129, 18944, 148 * 128 * 5 + 77, 262144 + 33, 1 << 20])
def test_pipeline_every_row_all_tile_shapes(env, mlp, cuda, n):
    """The pipeline over launches that end on full, partial and odd tiles and run 1..56 tiles per CTA, with HBM
    traffic on a second stream racing the kernel: every row within the bound of a torch fp64 forward pass, the
    penalty exact, the wrapping ring segment bit for bit against the dense output."""
    from flexgpu.predictor import DeviceReplayBuffer
    X = scenario_inputs(n, n, cuda)
    buf = DeviceReplayBuffer(n + 5, {"v_pred": 33, "safety_penalty": 1}, device=cuda)
    buf.reserve(n + 5)                                  # full ring: physical row = logical row
    pos = n // 3
    noise = torch.empty(256 << 20, dtype=torch.uint8, device=cuda)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        noise.add_(1)
    vhat, pen = mlp.predict(X, sink=buf, pos=pos)
    torch.cuda.synchronize()
    want, bound = forward_and_bound(mlp.weights, mlp.biases, "relu", X)
    assert bool(((vhat.double() - want).abs() <= bound).all())
    assert torch.allclose(pen, pen_ref(vhat, mlp), rtol=1e-12, atol=1e-9)
    assert int((pen > 0).sum()) > 0 or n < 1000
    idx = (pos + torch.arange(n, device=cuda)) % (n + 5)
    got = buf.get_batch(n + 5, start=0)
    assert torch.equal(got["v_pred"][idx], vhat) and torch.equal(got["safety_penalty"][idx, 0], pen.float())
    buf.close()


def test_replay_sink_with_wraparound(mlp, cuda):
    from flexgpu.predictor import DeviceReplayBuffer
    buf = DeviceReplayBuffer(1000, {"obs": 7, "v_pred": 33, "safety_penalty": 1}, device=cuda)
    ref = replay_ref.RefTransReplayBuffer(1000)
    for step in range(5):                                     # 5 x 300 rows into a 1000-row ring: wraps twice
        X = scenario_inputs(300, 100 + step, cuda, hi=1.3)
        obs = torch.rand(300, 7, device=cuda)
        pos = buf.reserve(300)
        buf.write("obs", pos, obs)
        vhat, pen = mlp.predict(X, sink=buf, pos=pos)
        ref.add_rows({"obs": obs.cpu().numpy(), "v_pred": vhat.cpu().numpy(), "safety_penalty": pen.float().cpu().numpy()[:, None]})
        assert len(buf) == len(ref) == min(1000, 300 * (step + 1))
    got = buf.get_batch(1000, start=0)
    for k in ("obs", "v_pred", "safety_penalty"):
        assert np.array_equal(got[k].cpu().numpy(), np.stack([t[k] for t in ref.buffer])), k
    buf.close()


def test_affine_and_mlp_coexist_on_one_handle(env, cuda):
    from flexgpu.predictor import MLPVoltagePredictor, VoltagePredictor
    rng = np.random.default_rng(21)
    pa = VoltagePredictor(env, rng.normal(0, 0.2, (33, 66)), rng.normal(1.0, 0.05, 33))
    X = torch.from_numpy(rng.uniform(-0.5, 0.5, (3000, 66)).astype(np.float32)).to(cuda)
    va, pa_ = pa.predict(X)                                   # the affine model alone
    W, b = random_mlp((64, 64), 22)
    pm = MLPVoltagePredictor(env, W, b, activation="tanh")
    vm, pm_ = pm.predict(X)
    assert env._resident_predictor is pa                      # loading the MLP did not evict the affine model
    for _ in range(2):
        v1, q1 = pa.predict(X)
        v2, q2 = pm.predict(X)
        assert torch.equal(v1, va) and torch.equal(q1, pa_) and torch.equal(v2, vm) and torch.equal(q2, pm_)
    launches = env.launch_count()
    pa.predict(X); pm.predict(X)
    assert env.launch_count() == launches + 2                 # no reload of either model between the calls


def test_argument_validation(env, cuda, profiles):
    from flexgpu import BatchedFlexProvisionEnv, FlexGpuError
    from flexgpu.predictor import DeviceReplayBuffer, MLPVoltagePredictor
    lib = env._lib

    def load(widths, act=1, v_min=0.9, v_max=1.1, w=1000.0, poison=None):
        W = [np.full((o, i), 0.01) for i, o in zip(widths[:-1], widths[1:])]
        Wf = np.concatenate([x.reshape(-1) for x in W]) if W else np.zeros(1)
        bf = np.zeros(max(1, sum(widths[1:])))
        if poison is not None:
            Wf[poison] = np.nan
        wi = (C.c_int32 * len(widths))(*widths)
        rc = lib.fp_predictor_load_mlp(env._h, len(widths) - 1, wi, Wf.ctypes.data_as(C.c_void_p), bf.ctypes.data_as(C.c_void_p),
                                       act, v_min, v_max, w)
        return rc, lib.fp_last_error(env._h).decode()

    for hidden in ((128, 128), (128, 64)):
        with pytest.raises(FlexGpuError, match="227 KB"):
            MLPVoltagePredictor(env, *random_mlp(hidden, 0))
    for shape in ((64,), (100,), (128,), (64, 64), (32, 32, 32)):
        assert load((66,) + shape + (33,))[0] == 0, shape
    bad = [dict(widths=(66, 16, 16, 16, 16, 33)), dict(widths=(66, 0, 33)), dict(widths=(66, 129, 33)),
           dict(widths=(65, 16, 33)), dict(widths=(66, 16, 32)), dict(widths=(66, 16, 33), poison=7),
           dict(widths=(66, 16, 33), act=4), dict(widths=(66, 16, 33), act=-1), dict(widths=(66, 16, 33), v_min=1.1, v_max=1.1),
           dict(widths=(66, 16, 33), w=0.0), dict(widths=(66, 16, 33), w=-1.0)]
    for kw in bad:
        rc, msg = load(**kw)
        assert rc == -1 and msg.startswith("fp_predictor_load_mlp:"), (kw, rc, msg)

    p = MLPVoltagePredictor(env, *random_mlp((16,), 1))
    with pytest.raises(ValueError):
        p.predict(torch.zeros(4, 65, device=cuda))
    flat = torch.zeros(11 * 66 + 1, device=cuda)
    with pytest.raises(FlexGpuError, match="16-byte"):
        p.predict(flat[1:].view(11, 66))                       # contiguous, 4 bytes past an aligned start
    buf = DeviceReplayBuffer(10, {"v_pred": 33}, device=cuda)
    with pytest.raises(FlexGpuError, match="replay ring"):
        p.predict(torch.zeros(11, 66, device=cuda), sink=buf, pos=0)     # more rows than the ring holds
    buf.close()

    fresh = BatchedFlexProvisionEnv(None, n_envs=8, device=cuda, profiles=profiles)   # nothing loaded yet
    X = torch.zeros(4, 66, device=cuda)
    assert lib.fp_predict_mlp(fresh._h, 4, C.c_void_p(X.data_ptr()), None, None, None, -1, -1, 0, None) == -3
    fresh.close()
