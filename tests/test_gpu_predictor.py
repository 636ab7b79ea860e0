"""GPU parity: the tcgen05 voltage predictor + safety penalty (fp_predict) and the device replay
ring (fp_replay_*) through the C ABI.

Tolerances: the kernel computes in 3xTF32 with fp32 accumulation and fp32 outputs, so Vhat is
compared with scikit-learn's fp64 predict at 1e-6 p.u. (north_star's voltage tolerance; observed
~2e-7) and the penalty at 1000 x 33 x that bound; ring contents are compared bit for bit with
the dense output."""
import os

import numpy as np
import pytest
import torch

from oracle import predictor_ref, replay_ref

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "predictor_golden.npz")
TOL_V = 1e-6


@pytest.fixture(scope="module")
def env(cuda, profiles):
    from flexgpu import BatchedFlexProvisionEnv
    e = BatchedFlexProvisionEnv(None, n_envs=8, device=cuda, profiles=profiles)
    yield e
    e.close()


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


@pytest.fixture(scope="module")
def pred(env, gold):
    from flexgpu.predictor import VoltagePredictor
    return VoltagePredictor.from_linear_model(env, gold["coef"], gold["intercept"], gold["x_scale"], gold["x_min"],
                                              gold["y_scale"], gold["y_min"])


def test_golden_vectors_sklearn_predict(pred, gold, cuda):
    X = torch.from_numpy(gold["X"].astype(np.float32)).to(cuda)
    vhat, pen = pred.predict(X)
    # the kernel sees fp32 inputs: compare with sklearn evaluated on the same rounded inputs
    want = predictor_ref.affine_predict(pred.A, pred.c, gold["X"].astype(np.float32).astype(np.float64))
    assert np.max(np.abs(vhat.cpu().numpy() - want)) < TOL_V
    assert np.max(np.abs(vhat.cpu().numpy() - gold["V"])) < 5e-6          # incl. the fp32 rounding of the inputs
    wantp = predictor_ref.slack_penalty(vhat.cpu().numpy().astype(np.float64))
    assert np.allclose(pen.cpu().numpy(), wantp, rtol=1e-12, atol=1e-9)    # fp64 penalty of the fp32 Vhat: exact arithmetic
    assert np.max(np.abs(pen.cpu().numpy() - gold["penalty"])) < 1000 * 33 * 5e-6
    assert int((pen == 0).sum()) >= 5 and float(pen.max()) > 1000.0


@pytest.mark.parametrize("n", [1, 2, 127, 128, 129, 255, 1000, 4097])
def test_ragged_sizes_and_random_models(env, cuda, n):
    """Odd sizes take the non-TMA tail path; every row depends only on its own inputs."""
    from flexgpu.predictor import VoltagePredictor
    rng = np.random.default_rng(n)
    A = rng.normal(0, 0.2, (33, 66)); c = rng.normal(1.0, 0.05, 33)
    p = VoltagePredictor(env, A, c)
    X = rng.uniform(-0.5, 0.5, (n, 66)).astype(np.float32)
    vhat, pen = p.predict(torch.from_numpy(X).to(cuda))
    want = predictor_ref.affine_predict(A, c, X.astype(np.float64))
    # 3xTF32 error model: the dropped lo*lo products and the truncated lo parts are each <= 2^-22 of
    # |a||x| per term, plus fp32 accumulation/bias rounding -> 2^-20 * (|A||x| + |c|) is a safe bound
    bound = 2.0 ** -20 * (np.abs(X.astype(np.float64)) @ np.abs(A).T + np.abs(c))
    assert vhat.shape == (n, 33) and np.all(np.abs(vhat.cpu().numpy() - want) <= bound)
    assert np.allclose(pen.cpu().numpy(), predictor_ref.slack_penalty(vhat.cpu().numpy().astype(np.float64)), rtol=1e-12, atol=1e-9)


def test_rowsum_quirk_form(env, gold, cuda):
    from flexgpu.predictor import VoltagePredictor
    p = VoltagePredictor.from_safemaddpg_rowsum(env, gold["coef"], gold["intercept"])
    X32 = gold["X"].astype(np.float32)
    vhat, _ = p.predict(torch.from_numpy(X32).to(cuda))
    want = predictor_ref.rowsum_predict(gold["coef"], gold["intercept"], X32.astype(np.float64))
    assert np.max(np.abs(vhat.cpu().numpy() - want)) < TOL_V * max(1.0, np.abs(want).max())


def test_epilogue_writes_straight_into_the_replay_ring_with_wraparound(pred, cuda):
    from flexgpu.predictor import DeviceReplayBuffer
    buf = DeviceReplayBuffer(1000, {"obs": 7, "v_pred": 33, "safety_penalty": 1}, device=cuda)
    ref = replay_ref.RefTransReplayBuffer(1000)
    rng = np.random.default_rng(0)
    for step in range(5):                                     # 5 x 300 rows into a 1000-row ring: wraps twice
        X = torch.from_numpy(rng.uniform(0, 0.6, (300, 66)).astype(np.float32)).to(cuda)
        obs = torch.from_numpy(rng.uniform(0, 1, (300, 7)).astype(np.float32)).to(cuda)
        pos = buf.reserve(300)
        buf.write("obs", pos, obs)
        vhat, pen = pred.predict(X, sink=buf, pos=pos)
        ref.add_rows({"obs": obs.cpu().numpy(), "v_pred": vhat.cpu().numpy(), "safety_penalty": pen.float().cpu().numpy()[:, None]})
        assert len(buf) == len(ref) == min(1000, 300 * (step + 1))
    got = buf.get_batch(1000, start=0)
    for k in ("obs", "v_pred", "safety_penalty"):
        want = np.stack([t[k] for t in ref.buffer])
        assert np.array_equal(got[k].cpu().numpy(), want), k
    np.random.seed(1); rs = np.random.RandomState(1)          # the reference's draw order (:17-18)
    for _ in range(5):
        b = buf.get_batch(64)
        wantb, start = ref.get_batch(64, rs)
        assert np.array_equal(b["v_pred"].cpu().numpy(), np.stack([t["v_pred"] for t in wantb]))
    buf.clear()
    assert len(buf) == 0
    with pytest.raises(ValueError):
        buf.get_batch(1)
    buf.close()


def test_config4_262144_envs_properties(env, pred, cuda):
    """BASELINE config 4 at full size: linearity of the affine map, sampled rows against fp64."""
    from flexgpu.predictor import DeviceReplayBuffer
    n = 262144
    g = torch.Generator(device=cuda).manual_seed(0)
    X = torch.rand(n, 66, device=cuda, generator=g) * 0.4
    buf = DeviceReplayBuffer(n, {"v_pred": 33, "safety_penalty": 1}, device=cuda)
    v1, p1 = pred.predict(X, sink=buf)
    v2, _ = pred.predict(2 * X)
    v0, _ = pred.predict(torch.zeros(4, 66, device=cuda))
    assert torch.allclose(v2 - v0[0], 2 * (v1 - v0[0]), rtol=0, atol=4e-6)            # affine: V(2x) - c = 2 (V(x) - c)
    idx = torch.arange(0, n, 4099, device=cuda)
    want = predictor_ref.affine_predict(pred.A, pred.c, X[idx].double().cpu().numpy())
    assert np.max(np.abs(v1[idx].cpu().numpy() - want)) < 2e-6
    got = buf.get_batch(n, start=0)
    assert torch.equal(got["v_pred"], v1) and torch.equal(got["safety_penalty"][:, 0], p1.float())
    buf.close()


def test_argument_validation(env, cuda):
    from flexgpu import FlexGpuError
    from flexgpu.predictor import DeviceReplayBuffer, VoltagePredictor
    with pytest.raises(FlexGpuError):
        VoltagePredictor(env, np.zeros((10, 20)), np.zeros(10))
    p = VoltagePredictor(env, np.zeros((33, 66)), np.ones(33))
    with pytest.raises(ValueError):
        p.predict(torch.zeros(4, 65, device=cuda))
    buf = DeviceReplayBuffer(10, {"v_pred": 33}, device=cuda)
    with pytest.raises(FlexGpuError):
        p.predict(torch.zeros(11, 66, device=cuda), sink=buf)     # more rows than the ring holds
    with pytest.raises(FlexGpuError):
        buf.reserve(0)
    buf.close()


@pytest.mark.parametrize("n", [127, 129, 18944, 148 * 128 * 5 + 77, 262144 + 33, 1 << 20])
def test_pipeline_every_row_all_tile_shapes(env, pred, cuda, n):
    """The warp-specialised pipeline (TMA ring of 4 tiles, two TMEM A buffers, two accumulators) over launches
    that end on full, partial and odd tiles and run 1..56 tiles per CTA, with HBM traffic on a second stream
    racing the kernel: EVERY row against a torch fp64 evaluation of the same affine map (1e-6 p.u.), the
    penalty against the fp64 formula on the returned Vhat (exact arithmetic), the ring segment (wrapping) bit
    for bit against the dense output."""
    from flexgpu.predictor import DeviceReplayBuffer
    from flexgpu import Network, create_network, DEFAULT_ENV_ARGS
    net = Network(create_network(DEFAULT_ENV_ARGS))
    base = torch.from_numpy(np.stack([net.base_p, net.base_q], axis=1).reshape(-1)).to(cuda)
    g = torch.Generator(device=cuda).manual_seed(n)
    X = (base[None, :] * (0.7 + 1.3 * torch.rand(n, 66, device=cuda, dtype=torch.float64, generator=g))).float().contiguous()
    A = torch.from_numpy(pred.A).to(cuda); c = torch.from_numpy(pred.c).to(cuda)
    buf = DeviceReplayBuffer(n + 5, {"v_pred": 33, "safety_penalty": 1}, device=cuda)
    buf.reserve(n + 5)                                  # full ring: physical row = logical row
    pos = n // 3
    noise = torch.empty(256 << 20, dtype=torch.uint8, device=cuda)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        noise.add_(1)
    vhat, pen = pred.predict(X, sink=buf, pos=pos)
    torch.cuda.synchronize()
    assert float((vhat.double() - (X.double() @ A.T + c)).abs().max()) < TOL_V
    vd = vhat.double()
    want = 1000.0 * (torch.clamp(pred.v_min - vd, min=0) + torch.clamp(vd - pred.v_max, min=0)).sum(dim=1)
    assert torch.allclose(pen, want, rtol=1e-12, atol=1e-9)
    assert int((pen > 0).sum()) > 0 or n < 1000          # the 2x-load scenarios leave the limits somewhere
    idx = (pos + torch.arange(n, device=cuda)) % (n + 5)
    got = buf.get_batch(n + 5, start=0)
    assert torch.equal(got["v_pred"][idx], vhat) and torch.equal(got["safety_penalty"][idx, 0], pen.float())
    buf.close()


# ---------------------------------------------------------------------------------------------------
# PINNED on the reference's own scripts (tests/golden/ref_predictor.npz, ref_replay.npz: made by
# safety_signal/data_generation.py, train_safety_signal_model.py and utils/replay_buffer.py themselves,
# tests/golden/make_ref_golden.py)
def test_reference_fit_predictions(env, cuda):
    """k_predict with the REFERENCE'S regressor + scalers against sklearn's predictions of all 1000 scenarios the
    reference generated, and against the scaled predictions its training script computed on its test split."""
    from flexgpu.predictor import VoltagePredictor
    from _golden import load_ref_predictor
    g = load_ref_predictor()
    p = VoltagePredictor.from_linear_model(env, g["coef"], g["intercept"], g["x_scale"], g["x_min"], g["y_scale"], g["y_min"])
    vhat, pen = p.predict(torch.from_numpy(g["X"].astype(np.float32)).to(cuda))
    V = vhat.cpu().numpy().astype(np.float64)
    assert np.max(np.abs(V - g["V_pred"])) < 2e-6               # 1e-6 kernel tolerance + the fp32 rounding of the inputs
    assert np.max(np.abs(V - g["Y"])) < 5e-3                    # ... and it does predict the power-flow voltages
    Xte = ((g["X_test_scaled"] - g["x_min"]) / g["x_scale"]).astype(np.float32)
    vte, _ = p.predict(torch.from_numpy(Xte).to(cuda))
    scaled = vte.cpu().numpy().astype(np.float64) * g["y_scale"] + g["y_min"]
    assert np.max(np.abs(scaled[:, 1:] - g["Y_pred_scaled"][:, 1:]) / g["y_scale"][1:]) < 2e-6   # back in p.u.
    want = predictor_ref.slack_penalty(V)
    assert np.allclose(pen.cpu().numpy(), want, rtol=1e-12, atol=1e-9)


def test_reference_replay_buffer_sequence(cuda):
    """DeviceReplayBuffer driven with the adds and the numpy seed that drove the reference's TransReplayBuffer:
    the same window starts (np.random.choice, :18) and the same transitions in every batch, FIFO eviction included."""
    from flexgpu.predictor import DeviceReplayBuffer
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_replay.npz"))
    buf = DeviceReplayBuffer(int(g["size"][0]), {"row": 7}, device=cuda)
    rows = torch.from_numpy(g["rows"]).to(cuda)
    np.random.seed(int(g["seed"][0]))
    n_added = 0
    for k, (n_target, batch) in enumerate(g["events"]):
        if n_target > n_added:
            buf.add_experience({"row": rows[n_added:n_target]}); n_added = int(n_target)
        got = buf.get_batch(int(batch))["row"].cpu().numpy()
        assert [int(x) for x in got[:, 0]] == list(g["ids"][k][:batch]), k
        assert np.array_equal(got, g["rows"][g["ids"][k][:batch]])
    assert len(buf) == len(g["final_ids"])
    assert [int(x) for x in buf.get_batch(len(buf), start=0)["row"][:, 0].cpu().numpy()] == list(g["final_ids"])
    buf.close()
