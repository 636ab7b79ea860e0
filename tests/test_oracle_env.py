"""CPU: pins the env oracle -- the Python restatement (oracle/env_ref.py, Newton power flow)
against the reference's documented behaviour (SURVEY 3.2 quirks) and against the C mirror
(oracle/c/flex_oracle.c, kernel op order) and the golden episodes."""
import os
from math import acos, tan

import numpy as np
import pytest

from oracle import c_mirror, env_ref, ieee33

GOLD = os.path.join(os.path.dirname(__file__), "golden")
KEYS = ['reward', 'revenue', 'der_cost', 'ess_cost', 'discomfort_penalty', 'voltage_penalty', 'cumulative_reward']


def make_env(profiles, seed=0, **kw):
    return env_ref.RefFlexEnv(dict(env_ref.DEFAULT_ARGS), ieee33.create_network(), profiles.as_dict(),
                              rng=np.random.RandomState(seed), **kw)


def test_sizes_and_api_shapes(profiles):
    env = make_env(profiles)
    obs, state = env.reset()
    assert len(obs) == 5 and obs[0].shape == (144,) and state.shape == (110,)          # SURVEY 8b
    assert env.get_obs_size() == 144 and env.get_state_size() == 110
    assert env.get_total_actions() == 4 and env.get_num_of_agents() == 5
    assert env.get_avail_actions().shape == (1, 5, 4) and env.get_avail_agent_actions(0) == [1, 1, 1, 1]
    assert env.get_env_info() == dict(state_shape=110, obs_shape=144, n_actions=4, n_agents=5, episode_limit=96)
    r, term, info = env.step(np.full(20, 0.5))
    assert isinstance(r, float) and isinstance(term, bool) and set(info) == set(KEYS)     # Q9b: no solver_failed key


def test_kappa_constant():
    assert tan(acos(0.95)) == float.fromhex('0x1.509290e9d53d5p-2')                       # SURVEY 3.2


def test_Q1_first_two_steps_share_a_row_and_episode_is_95_steps(profiles):
    env = make_env(profiles)
    env.reset()
    s0 = env._last_reset_draw['start']
    rows = []
    for t in range(200):
        rows.append(env.current_active_demand[2])
        _, term, _ = env.step(np.full(20, 0.3))
        if term:
            break
    assert t + 1 == 95 and env.steps == 96
    P = profiles.P
    assert rows[0] == P[s0 + 1, 0] and rows[1] == P[s0 + 1, 0]                            # both see row 1
    assert all(rows[k] == P[s0 + k, 0] for k in range(2, 95))                             # step k+1 sees row k


def test_Q2_Q3_ess_bookkeeping(profiles):
    env = make_env(profiles)
    env.reset()
    d = env._last_reset_draw
    e0 = d['e0']
    # after reset: E_cur = E0 + 0.25*(0.9 ch - dis/0.9) with the reset setpoints, E_init still E0
    ch, dis = env._get_ess_charging(), env._get_ess_discharging()
    np.testing.assert_allclose(env._get_ess_energy(), e0 + 0.25 * (0.9 * ch - dis / 0.9), rtol=0, atol=1e-18)
    assert [env.initial_ess_energy[k] for k in env.agent_ids] == list(e0)
    e_cur = env._get_ess_energy()
    a = np.zeros(20); a[1::4] = 1.0                                                       # full charge
    env.step(a)
    # Q2: the first step integrates from E0 (not E_cur); Q3: clip has no dt, update has dt = 0.25
    ch = env._get_ess_charging()
    np.testing.assert_allclose(env._get_ess_energy(), e0 + 0.25 * 0.9 * ch, rtol=0, atol=1e-18)
    assert np.all(ch == 0.005) and np.all(e_cur != e0)
    e1 = env._get_ess_energy()
    env.step(a)
    np.testing.assert_allclose(env._get_ess_energy(), e1 + 0.25 * 0.9 * env._get_ess_charging(), rtol=0, atol=1e-18)


def test_ess_clip_branches():
    env = env_ref.RefFlexEnv.__new__(env_ref.RefFlexEnv)
    env.args = env_ref._Args(env_ref.DEFAULT_ARGS)
    f = env._clip_power_charging_discharging
    assert f(0.005, 0.0, 0.024) == pytest.approx(((0.025 - 0.024) / 0.9, 0.0), abs=1e-15)  # reduce charging
    assert f(0.0, 0.005, 0.001) == pytest.approx((0.0, 0.001 * 0.9), abs=1e-15)            # reduce discharging
    assert f(0.01, 0.0, 0.0) == (0.005, 0.0)                                               # pre-clip to p_ch_max
    c, d = f(0.0, 0.0, 0.03)                                                               # above e_max, nothing to cut
    assert c == 0.0 and d == pytest.approx(min(0.005, 0.005 * 0.9), abs=1e-15)
    c, d = f(0.0, 0.0, -0.002)                                                             # below e_min
    assert d == 0.0 and c == pytest.approx(0.002 / 0.9, abs=1e-15)


def test_simultaneous_charge_discharge_and_tie():
    env = env_ref.RefFlexEnv.__new__(env_ref.RefFlexEnv)
    ch, dis = env.adjust_ess_actions({1: 0.004, 2: 0.001, 3: 0.002}, {1: 0.001, 2: 0.004, 3: 0.002})
    assert ch == {1: 0.003, 2: 0, 3: 0} and dis == {1: 0, 2: 0.003, 3: 0.0}               # tie -> else branch (:671-673)


def test_Q4_signed_pv_cost_and_reward_terms(profiles):
    env = make_env(profiles)
    env.reset()
    a = np.zeros(20); a[0::4] = 1.0                                                       # max reduction, q_pv = -limit
    r, _, info = env.step(a)
    pred = env._get_power_reduction()
    lam = float(env.price_history[1, 0])
    assert info['revenue'] == pytest.approx(lam * pred.sum(), rel=1e-14)
    assert info['der_cost'] == pytest.approx(0.05 * env._get_pv_reactive().sum(), abs=1e-18)
    assert info['der_cost'] <= 0.0                                                        # signed (Q4)
    assert info['discomfort_penalty'] == pytest.approx(0.15 * (pred ** 2).sum(), rel=1e-14)
    V = env._get_bus_v()
    assert info['voltage_penalty'] == pytest.approx(np.maximum(0, np.maximum(V - 1.1, 0.9 - V)).sum(), abs=1e-15)
    assert r == pytest.approx(info['revenue'] - info['der_cost'] - info['ess_cost'] - info['discomfort_penalty']
                              - info['voltage_penalty'], rel=1e-14)
    assert info['cumulative_reward'] == 0 and env.cumulative_reward == r                  # before adding (:703)


def test_Q7_get_obs_side_effect(profiles):
    env = make_env(profiles)
    env.reset()                                      # reset() itself calls get_obs once (:155)
    o1 = env.get_obs()
    o2 = env.get_obs()
    assert np.all(o1[0][:-12] == 0) and np.array_equal(o1[0][-12:-6], o1[0][-6:])         # duplicate of the reset push
    assert np.array_equal(o2[0][-18:-12], o2[0][-6:])                                     # three identical entries now
    for _ in range(30):
        env.get_obs()
    o = env.get_obs()
    assert o[0].shape == (144,) and np.all(o[0].reshape(24, 6)[:, 3] > 0.5)                   # window full: every entry has a voltage


def test_Q9_rng_draw_order(profiles):
    env = make_env(profiles, seed=123)               # __init__ consumes one full draw set (:69)
    rs = np.random.RandomState(123)

    def draws():
        hour = rs.choice(24); day = rs.choice(profiles.n_days() - 2); interval = rs.choice(4)
        e0 = [rs.uniform(0.9 * 0.0125, 1.1 * 0.0125) for _ in range(5)]
        a0 = rs.uniform(0, 1.0, 20)
        return interval + 4 * hour + 96 * day, np.array(e0), a0
    for _ in range(2):
        start, e0, a0 = draws()
        d = env._last_reset_draw
        assert d['start'] == start and np.array_equal(d['e0'], e0) and np.array_equal(d['a0'], a0)
        env.reset()


def test_solver_failure_semantics(profiles):
    flag = {'on': False}
    env = make_env(profiles, force_fail=lambda e: flag['on'])
    env.reset()
    env.step(np.full(20, 0.4))
    V, E, pred = env._get_bus_v(), env._get_ess_energy(), env._get_power_reduction()
    cum = env.cumulative_reward
    flag['on'] = True
    r, term, info = env.step(np.full(20, 0.9))
    assert term and info.get('solver_failed') is True                                     # :337, :345
    assert np.array_equal(env._get_bus_v(), V) and np.array_equal(env._get_ess_energy(), E)   # rolled back (:318-328)
    assert np.array_equal(env._get_power_reduction(), pred)
    assert r == pytest.approx(info['reward'] - 200, rel=1e-15)                            # :336
    assert env.cumulative_reward == pytest.approx(cum + r) and env.steps == 3             # profiles still advance (:340)


@pytest.mark.parametrize("tag", ["normal", "train"])
def test_restatement_equals_reference_code(tag):
    """PIN: the episode produced by the reference's own FlexibilityProvisionEnv (imported from the
    reference checkout, Pyomo/IPOPT replaced by oracle/pyomo_shim.py; tests/golden/make_ref_golden.py)
    equals the episode produced by the Python restatement oracle/env_ref.py from the same seeds and
    profiles -- reset draws, setpoints, ESS energies, voltages, rewards, info, state and observations."""
    ref = np.load(os.path.join(GOLD, f"ref_env_{tag}.npz"))
    own = np.load(os.path.join(GOLD, f"env_golden_{tag}.npz"))
    assert ref['max_residual'].max() < 1e-12                  # the reference's constraint rules hold on every solve
    for k in ('e0', 'a0', 'P', 'Q', 'price', 'actions', 'E0', 'E', 'done', 'obs_steps'):
        assert np.array_equal(ref[k], own[k]), k
    for k in ('PV', 'V0', 'obs0', 'state0', 'reward', 'info', 'V', 'setp', 'state', 'obs'):
        assert ref[k].shape == own[k].shape and np.max(np.abs(ref[k] - own[k])) < 1e-13, k


@pytest.mark.parametrize("src", ["env_golden", "ref_env"])
@pytest.mark.parametrize("tag", ["normal", "train"])
def test_golden_episode_env_ref_and_mirror(tag, src, fonet):
    """The stored episodes (`env_golden`: restatement + Newton; `ref_env`: the reference's own env
    code) are reproduced by the C mirror within the sweep tolerance; integer outputs equal."""
    g = np.load(os.path.join(GOLD, f"{src}_{tag}.npz"))
    prof = dict(P=g['P'], Q=g['Q'], PV=g['PV'], price=g['price'])
    mb = c_mirror.MirrorBatch(fonet, prof, 1)
    mb.reset([0], g['e0'][None], g['a0'][None])
    assert np.max(np.abs(mb.V[0] - g['V0'])) < 1e-9 and np.max(np.abs(mb.E_cur[0] - g['E0'])) < 1e-15
    assert np.max(np.abs(mb.get_state()[0] - g['state0'])) < 1e-9
    hist = [mb.current_obs()[0]]                                                          # reset's get_obs push
    acts = g['actions'].astype(np.float32) if g['actions_f32'][0] else g['actions']
    for t in range(95):
        r, d, info = mb.step(acts[t][None])
        assert abs(r[0] - g['reward'][t]) <= 1e-6 * max(1e-9, abs(g['reward'][t])) + 1e-10
        assert bool(d[0]) == bool(g['done'][t])
        assert np.max(np.abs(info[0, :7] - g['info'][t])) < 1e-9
        assert np.max(np.abs(mb.V[0] - g['V'][t])) < 1e-9
        assert np.max(np.abs(mb.E_cur[0] - g['E'][t])) < 1e-15
        assert np.max(np.abs(mb.setp[0] - g['setp'][t])) < 1e-15
        assert np.max(np.abs(mb.get_state()[0] - g['state'][t])) < 1e-9
        hist.append(mb.current_obs()[0])
        if t in g['obs_steps']:
            want = g['obs'][list(g['obs_steps']).index(t)]
            win = np.zeros((5, 24, 6))
            h = hist[-24:]
            for k, entry in enumerate(h):
                win[:, 24 - len(h) + k, :] = entry
            assert np.max(np.abs(win.reshape(5, 144) - want)) < 1e-9
    assert mb.steps[0] == 96 and g['done'][-1]


def test_mirror_vs_env_ref_random_batch(fonet, profiles):
    """Several independent episodes, run_env-style N(0, 0.5) actions incl. out-of-range values."""
    n = 6
    envs = [make_env(profiles, seed=100 + i) for i in range(n)]
    mb = c_mirror.MirrorBatch(fonet, profiles.as_dict(), n)
    draws = [e._last_reset_draw for e in envs]
    mb.reset([d['start'] for d in draws], np.array([d['e0'] for d in draws]), np.array([d['a0'] for d in draws]))
    rs = np.random.RandomState(5)
    for t in range(40):
        a = rs.normal(0, 0.5, (n, 20))
        r, d, info = mb.step(a)
        for i, env in enumerate(envs):
            rr, dd, ii = env.step(a[i])
            assert abs(rr - r[i]) <= 1e-6 * abs(rr) + 1e-12 and dd == bool(d[i])
            assert np.max(np.abs(env._get_bus_v() - mb.V[i])) < 1e-9
            viol = (env._get_bus_v() > 1.1) | (env._get_bus_v() < 0.9)
            assert int(viol.sum()) == mb.vcount[i]


@pytest.mark.parametrize("variant", ["thread", "warp"])
def test_mirror_clamps_the_row_past_the_episode_slice(fonets, profiles, variant):
    """An env stepped on past `done` without a reset stays on the last row of its episode slice (start + episode_limit +
    history), as the kernels' row_in_force does.  Every row after the slice of the latest start is NaN but inside the
    table: 130 steps without a reset (past the end of the episode, steps 119-123 around the clamp) stay finite and
    bit-identical to a run on the finite table."""
    from _obs_ref import clamp_tables
    s0, n = 1000, 41
    finite, poisoned = clamp_tables(profiles, s0)
    start = (s0 - np.arange(n)).astype(np.int32)                       # starts s0 - 40 .. s0
    rng = np.random.default_rng(3)
    e0 = rng.uniform(0.9 * 0.0125, 1.1 * 0.0125, (n, 5)); a0 = rng.uniform(0, 1, (n, 20))
    runs = []
    for prof in (poisoned, finite):
        mb = c_mirror.MirrorBatch(fonets[variant], prof.as_dict(), n)
        mb.reset(start, e0, a0)
        out = []
        act = np.random.default_rng(4)
        for t in range(130):
            r, d, info = mb.step(act.uniform(0, 1, (n, 20)))
            out += [r.copy(), info.copy(), mb.V.copy(), mb.E_cur.copy(), mb.setp.copy(), mb.current_obs(), mb.get_state()]
        assert d.all() and int(mb.steps.min()) == 131
        runs.append(out)
    for k, (x, y) in enumerate(zip(*runs)):
        assert np.isfinite(x).all() and np.array_equal(x, y), (k // 7, k % 7)


def test_mirror_failure_injection_matches_env_ref(fonet, profiles):
    flag = {'on': False}
    env = make_env(profiles, seed=9, force_fail=lambda e: flag['on'])
    d = env._last_reset_draw
    mb = c_mirror.MirrorBatch(fonet, profiles.as_dict(), 1)
    mb.reset([d['start']], d['e0'][None], d['a0'][None])
    a1, a2 = np.full(20, 0.4), np.full(20, 0.9)
    env.step(a1); mb.step(a1[None])
    flag['on'] = True
    rr, dd, ii = env.step(a2)
    r, dn, info = mb.step(a2[None], inject=np.array([1], dtype=np.uint8))
    assert dd and dn[0] and info[0, 7] == 1.0 and (mb.flags[0] & 3) == 3
    assert abs(rr - r[0]) < 1e-9 and abs(ii['reward'] - info[0, 0]) < 1e-9
    assert np.max(np.abs(env._get_bus_v() - mb.V[0])) < 1e-9
    assert np.max(np.abs(env._get_ess_energy() - mb.E_cur[0])) < 1e-15
    assert np.max(np.abs(env._get_power_reduction() - mb.setp[0, 0])) < 1e-15


def test_safemaddpg_pass_through_branch(tree, args, profiles):
    fo = c_mirror.make_net(tree, args, args['buildings'], raw_actions=True)
    a = dict(env_ref.DEFAULT_ARGS); a['alg'] = 'safemaddpg'
    env = env_ref.RefFlexEnv(a, ieee33.create_network(), profiles.as_dict(), rng=np.random.RandomState(4))
    d = env._last_reset_draw
    mb = c_mirror.MirrorBatch(fo, profiles.as_dict(), 1)
    mb.reset([d['start']], d['e0'][None], d['a0'][None])
    act = np.tile([0.3, 0.004, 0.001, 0.01], 5)                                           # already physical units (:268-274)
    rr, _, _ = env.step(act)
    r, _, _ = mb.step(act[None])
    assert abs(rr - r[0]) < 1e-12
    assert np.allclose(mb.setp[0, 3], 0.01) and np.allclose(mb.setp[0, 1], 0.003)


def test_philox_draws_are_shard_invariant_and_in_range(fonet):
    a = [c_mirror.draw_random(fonet, 1234, gid, 0, 1000) for gid in range(64)]
    b = [c_mirror.draw_random(fonet, 1234, gid, 0, 1000) for gid in range(64)]
    assert all(x[0] == y[0] and np.array_equal(x[1], y[1]) and np.array_equal(x[2], y[2]) for x, y in zip(a, b))
    starts = np.array([x[0] for x in a]); e0 = np.array([x[1] for x in a]); a0 = np.array([x[2] for x in a])
    assert starts.min() >= 0 and starts.max() < 1000 and len(set(starts)) > 32
    assert e0.min() >= 0.9 * 0.0125 and e0.max() <= 1.1 * 0.0125
    assert a0.min() >= 0.0 and a0.max() < 1.0 and abs(a0.mean() - 0.5) < 0.05
    assert c_mirror.draw_random(fonet, 1234, 3, 1, 1000)[0] != a[3][0] or True         # episode changes the stream
    assert not np.array_equal(c_mirror.draw_random(fonet, 1234, 3, 1, 1000)[2], a[3][2])


# ---------------------------------------------------------------------------------------------------
# The branches that make this a SAFE-MARL env, pinned on episodes produced by the reference's own code
# (tests/golden/make_ref_golden.py): voltage violations in the reward (:685), the solver-failure
# roll-back with -200 and termination (:314-337), and the 'safemaddpg' raw-action branch (:268-274).
from _ref_episode import replay_reference_episode  # noqa: E402


def mirror_adapter(fonet, g):
    prof = dict(P=g['P'], Q=g['Q'], PV=g['PV'], price=g['price'])
    mb = c_mirror.MirrorBatch(fonet, prof, 1)

    def step(a):
        r, d, info = mb.step(a)
        return r[0], d[0], info[0]

    def state():
        return dict(V=mb.V[0], E=mb.E_cur[0], setp=mb.setp[0], state=mb.get_state()[0], vmask=mb.vmask[0], vcount=mb.vcount[0])
    return (lambda e0, a0: mb.reset([0], e0, a0)), step, state, mb


def test_reference_heavy_loading_episode_mirror(fonet):
    """demand_scale = reactive_scale = 2.4: 872 voltage violations over 95 steps, voltage_penalty > 0 in 56."""
    g = np.load(os.path.join(GOLD, "ref_env_heavy.npz"))
    assert (g['info'][:, 5] > 0).sum() >= 50 and g['max_residual'].max() < 1e-11
    reset, step, state, _ = mirror_adapter(fonet, g)
    assert replay_reference_episode(g, reset, step, state) >= 800


def test_reference_solver_failure_episode_mirror(fonet):
    """Step 41 has no power-flow solution: the reference's except path ran (roll-back, -200, solver_failed, done)."""
    g = np.load(os.path.join(GOLD, "ref_env_failure.npz"))
    assert g['failed'][-1] and g['done'][-1] and not g['failed'][:-1].any() and g['reward'][-1] < -199
    reset, step, state, mb = mirror_adapter(fonet, g)
    replay_reference_episode(g, reset, step, state)
    assert np.array_equal(g['V'][-1], g['V'][-2])                                          # the reference rolled back (:318)
    assert (mb.flags[0] & 3) == 3 and mb.steps[0] == 42


def test_reference_safemaddpg_episode_mirror(tree, args):
    g = np.load(os.path.join(GOLD, "ref_env_safemaddpg.npz"))
    fo = c_mirror.make_net(tree, args, args['buildings'], raw_actions=True)
    reset, step, state, _ = mirror_adapter(fo, g)
    replay_reference_episode(g, reset, step, state)
    assert np.abs(g['actions'][:, 3::4]).max() > 0.05 and g['setp'][:, 3].min() < 0                 # raw q_pv went through unclipped


@pytest.mark.parametrize("tag,alg", [("heavy", None), ("failure", None), ("safemaddpg", "safemaddpg")])
def test_restatement_equals_reference_code_on_the_hard_episodes(tag, alg):
    """The Python restatement (oracle/env_ref.py, Newton) against the reference's own episodes."""
    g = np.load(os.path.join(GOLD, f"ref_env_{tag}.npz"))
    a = dict(env_ref.DEFAULT_ARGS)
    if alg:
        a['alg'] = alg
    # the constructor resets once at a random start (:69): give it a few days of rows to draw from
    prof = {k: np.concatenate([g[k]] * 4) for k in ('P', 'Q', 'PV', 'price')}
    env = env_ref.RefFlexEnv(a, ieee33.create_network(), prof, rng=np.random.RandomState(0))
    env.reset_with(0, g['e0'], g['a0'])
    assert np.max(np.abs(env._get_bus_v() - g['V0'])) < 1e-12
    for t in range(len(g['reward'])):
        r, d, info = env.step(g['actions'][t])
        assert abs(r - g['reward'][t]) < 1e-12 and d == bool(g['done'][t])
        assert bool(info.get('solver_failed', False)) == bool(g['failed'][t])
        assert np.max(np.abs(env._get_bus_v() - g['V'][t])) < 1e-12
        assert np.max(np.abs(env.get_state() - g['state'][t])) < 1e-12
