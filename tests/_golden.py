"""Compact storage of the two largest reference fixtures (tests/golden/ref_policy.npz, ref_predictor.npz).

Inputs the reference's generators drew from seeded numpy streams (observation windows, Transitions, load
scenarios), and arrays that are plain rearrangements of them (the unpack_data batch, the critic input), are not
stored: `load_ref_policy()` / `load_ref_predictor()` redraw or rebuild them and check each one against the
SHA-256 of the reference's own bytes, stored beside the data, so the tests compare with exactly what the
reference produced.  The recurrent hidden states are stored for a fixed seeded subset of the envs
(`hid_rows`); every other output is stored for all of them."""
import hashlib
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
N_ENVS, NA, OBS, ACT, HID, STEPS = 160, 5, 144, 4, 64, 3
N_TRANSITIONS, BUFFER, BATCH = 80, 64, 32
HID_ROWS = 48
TR_FIELDS = ("state", "action", "log_prob_a", "value", "next_value", "reward", "next_state", "done", "last_step",
             "action_avail", "last_hid", "hid")


def digest(a):
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def _checked(name, a, stored):
    if digest(a) != str(stored["sha256_" + name]):
        raise AssertionError(f"rebuilt {name} differs from the reference's bytes (numpy stream or layout changed)")
    return a


# ------------------------------------------------------------------------------------------------- policy
def policy_windows(rng, n):
    """make_ref_policy_golden.windows: observation windows of the env's shape and magnitudes."""
    o = np.zeros((n, NA, 24, 6), dtype=np.float64)
    o[..., 0] = rng.uniform(0.02, 0.3, (n, NA, 24)); o[..., 1] = rng.uniform(0.005, 0.2, (n, NA, 24))
    o[..., 2] = rng.uniform(0.0, 0.15, (n, NA, 24)); o[..., 3] = rng.uniform(0.9, 1.02, (n, NA, 24))
    o[..., 4] = rng.uniform(0.05, 0.3, (n, NA, 24)); o[..., 5] = rng.uniform(0.0, 0.025, (n, NA, 24))
    pad = rng.integers(0, 24, n)
    for e in range(n):
        o[e, :, :pad[e] // 3] = 0.0
    return o.reshape(n, NA, OBS).astype(np.float32)


def policy_transitions():
    """The 80 Transitions make_ref_policy_golden.py adds to TransReplayBuffer(64), in its draw order, flattened."""
    rs = np.random.RandomState(3)
    rows = {k: [] for k in TR_FIELDS}
    for _ in range(N_TRANSITIONS):
        state = [rs.uniform(-1, 1, OBS) for _ in range(NA)]
        nstate = [rs.uniform(-1, 1, OBS) for _ in range(NA)]
        tr = dict(action=rs.uniform(-1, 1, (1, NA, ACT)).astype(np.float32), log_prob_a=rs.uniform(-3, 0, (1, NA, ACT)).astype(np.float32),
                  value=rs.uniform(-1, 1, (1, NA, 1)).astype(np.float32), next_value=rs.uniform(-1, 1, (1, NA, 1)).astype(np.float32),
                  reward=np.array([rs.uniform(-2, 2)] * NA))
        tr.update(state=state, next_state=nstate, done=bool(rs.rand() < 0.1), last_step=bool(rs.rand() < 0.1),
                  action_avail=np.ones((1, NA, ACT), dtype=np.int64))
        tr.update(last_hid=rs.uniform(-1, 1, (1, NA, HID)).astype(np.float32), hid=rs.uniform(-1, 1, (1, NA, HID)).astype(np.float32))
        for k in TR_FIELDS:
            rows[k].append(np.asarray(tr[k], dtype=np.float64).reshape(-1))
    return {"tr_" + k: np.stack(v).astype(np.float32) for k, v in rows.items()}


def _policy_batch(tr, start):
    """The rows get_batch(32) returns (the FIFO holds the last 64 adds) as unpack_data shapes them, and the critic
    input MADDPG.value builds from them: per (batch row, agent i) [obs of all agents | one-hot(i) | all actions]."""
    rows = slice(N_TRANSITIONS - BUFFER + start, N_TRANSITIONS - BUFFER + start + BATCH)
    up = {"up_" + k: tr["tr_" + k][rows].reshape(BATCH, NA, -1) for k in ("state", "next_state", "last_hid", "hid")}
    obs_all = up["up_state"].reshape(BATCH, 1, NA * OBS).repeat(NA, axis=1)
    act_all = tr["tr_action"][rows].reshape(BATCH, 1, NA * ACT).repeat(NA, axis=1)
    eye = np.broadcast_to(np.eye(NA, dtype=np.float32), (BATCH, NA, NA))
    up["critic_in"] = np.concatenate([obs_all, eye, act_all], axis=-1).reshape(BATCH * NA, -1)
    return up


def _policy_rebuilt(stored):
    rng = np.random.default_rng(0)
    out = {f"obs{t}": policy_windows(rng, N_ENVS) for t in range(STEPS)}
    out.update(policy_transitions())
    out.update(_policy_batch(out, int(stored["batch_start"])))
    return out


def compact_ref_policy(full):
    """What ref_policy.npz stores, from the complete set of arrays make_ref_policy_golden.py records."""
    out = {k: v for k, v in full.items()}
    rebuilt = _policy_rebuilt(full)
    for k, v in rebuilt.items():
        assert np.array_equal(v, full[k]) and v.dtype == full[k].dtype, k
        out["sha256_" + k] = np.array(digest(full[k]))
        del out[k]
    rows = np.sort(np.random.default_rng(0).choice(N_ENVS, HID_ROWS, replace=False))
    for t in range(STEPS):
        for tag in ("", "t_"):
            out[f"{tag}hid{t}"] = np.ascontiguousarray(full[f"{tag}hid{t}"][rows])
    out["hid_rows"] = rows
    return out


def load_ref_policy():
    stored = dict(np.load(os.path.join(GOLDEN, "ref_policy.npz")))
    for k, v in _policy_rebuilt(stored).items():
        stored[k] = _checked(k, v, stored)
    return stored


# ------------------------------------------------------------------------------------------------- predictor
def predictor_scenarios(n=1000, seed=2024, variation=0.3):
    """The load scenarios safety_signal/data_generation.py draws (numpy's global stream seeded with 2024): per scenario
    33 P then 33 Q factors on the IEEE 33-bus base loads, interleaved [P1, Q1, P2, Q2, ...]."""
    from oracle.ieee33 import create_network
    net = create_network()
    P0 = np.array([net["active_power_demand"][b] for b in net["bus_numbers"]])
    Q0 = np.array([net["reactive_power_demand"][b] for b in net["bus_numbers"]])
    rs = np.random.RandomState(seed)
    X = []
    for _ in range(n):
        p = P0 * (1 + rs.uniform(-variation, variation, len(P0)))
        q = Q0 * (1 + rs.uniform(-variation, variation, len(Q0)))
        X.append(np.stack([p, q], axis=1).reshape(-1))
    return np.array(X)


def compact_ref_predictor(full):
    out = {k: v for k, v in full.items() if k != "X"}
    assert np.array_equal(predictor_scenarios(len(full["X"])), full["X"])
    out["sha256_X"] = np.array(digest(full["X"]))
    return out


def load_ref_predictor():
    stored = dict(np.load(os.path.join(GOLDEN, "ref_predictor.npz")))
    stored["X"] = _checked("X", predictor_scenarios(len(stored["Y"])), stored)
    return stored
