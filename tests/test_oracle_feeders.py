"""CPU: the feeder catalogue of tests/_feeders.py sits where its table says (chains, slots, depth, thread shape), the C
mirror agrees with dense Newton on every catalogue feeder in both kernel variants' operation orders, and the fp64
restatement of the env runs an episode on each of them."""
import numpy as np
import pytest

import _feeders as F
from oracle import c_mirror, env_ref, ieee33, pf_ref


@pytest.mark.parametrize("name", list(F.CATALOGUE))
def test_catalogue_entry_reaches_its_row(name):
    net = F.feeder(name)
    _, want, shape, thread_ok = F.CATALOGUE[name]
    tree = ieee33.tree_arrays(net)
    assert len(net['bus_numbers']) == want["nb"] and len(net['buildings']) == want["na"]
    got = F.tree_counts(tree['parent'])
    assert got == {k: want[k] for k in ("chains", "slots", "depth")}, got
    assert F.thread_shape(net) == shape
    assert thread_ok == (got["chains"] <= F.MAX_CHAINS and got["slots"] <= F.MAX_SLOTS)
    assert 2 <= want["nb"] <= 33 and 1 <= want["na"] <= 5


def test_catalogue_covers_the_limits():
    rows = {n: F.CATALOGUE[n][1] for n in F.CATALOGUE}
    assert rows["limits_16x8"]["chains"] == F.MAX_CHAINS and rows["limits_16x8"]["slots"] == F.MAX_SLOTS
    assert rows["over_17_chains"]["chains"] == F.MAX_CHAINS + 1 and rows["over_9_slots"]["slots"] == F.MAX_SLOTS + 1
    assert rows["chain33"]["depth"] == 31                     # 5 pointer-jumping rounds cover 1 + 2 + 4 + 8 + 16 ancestors
    assert rows["two_bus"]["nb"] == 2
    star = ieee33.tree_arrays(F.feeder("slack_star"))
    assert int((star['parent'] == 0).sum()) >= 6
    assert F.thread_shape(ieee33.create_network()) == F.SHAPE_IEEE33   # the selection rule's positive case
    assert {F.CATALOGUE[n][1]["na"] for n in F.CATALOGUE} >= {1, 2, 3, 4, 5}
    resc = F.feeder("ieee33_rescaled")
    assert not any(v > 0 for v in resc['max_line_currents'].values())  # any_imax = 0
    base = ieee33.create_network()
    assert all(abs(resc['line_resistances'][k] - 1.7 * base['line_resistances'][k]) <= 1e-15 for k in base['line_connections'])
    perm = F.feeder("ieee33_permuted")
    assert perm['bus_numbers'][0] == 1 and perm['bus_numbers'] != sorted(perm['bus_numbers'])
    assert any((t, f) in base['line_resistances'] for (f, t) in perm['line_connections'])


def test_lindistflow_map_is_the_ieee33_one_and_linearises_the_power_flow():
    """On IEEE-33 the builder gives the map the safety-affine tests use; on every feeder it predicts the solved voltages
    to first order at light load."""
    for name in F.CATALOGUE:
        net = F.feeder(name)
        tree = ieee33.tree_arrays(net)
        A, c = F.lindistflow_map(tree)
        nb = len(tree['parent'])
        assert A.shape == (nb, 2 * nb) and c.shape == (nb,)
        assert not A[0].any() and not A[:, 0:2].any()                 # the slack bus: fixed voltage, no injection
        p = np.array([net['active_power_demand'][b] for b in net['bus_numbers']]) * 0.05
        q = np.array([net['reactive_power_demand'][b] for b in net['bus_numbers']]) * 0.05
        sol = pf_ref.solve_newton(tree, p, q)
        x = np.empty(2 * nb); x[0::2] = p; x[1::2] = q
        v2 = A @ (2 * x) + c                                          # LinDistFlow in squared voltages: v = 1 - 2 (R P + X Q)
        assert np.max(np.abs(v2 - sol['v'])) < 1e-4, name


@pytest.mark.parametrize("variant", [c_mirror.VARIANT_THREAD, c_mirror.VARIANT_WARP])
@pytest.mark.parametrize("name", list(F.CATALOGUE))
def test_mirror_matches_newton_on_every_feeder(name, variant):
    """200 random loadings (0.5x - 1.6x per bus): V, P, Q within 1e-8 p.u. and line currents within 1e-7 p.u., the bars
    the IEEE-33 power-flow tests hold (the thread variant stops on |dl| <= 1e-5, so a squared current of ~20 p.u. on a
    loaded trunk head is ~2e-7 off while its current is inside 1e-7)."""
    net = F.feeder(name)
    tree = ieee33.tree_arrays(net)
    fon = c_mirror.make_net(tree, F.env_args(net), net['buildings'], variant=variant)
    nb = len(tree['parent'])
    base_p = np.array([net['active_power_demand'][b] for b in net['bus_numbers']])
    base_q = np.array([net['reactive_power_demand'][b] for b in net['bus_numbers']])
    rng = np.random.default_rng(7)
    p = base_p[None, 1:] * rng.uniform(0.5, 1.6, (200, nb - 1))
    q = base_q[None, 1:] * rng.uniform(0.5, 1.6, (200, nb - 1))
    out = c_mirror.mirror_power_flow(fon, p, q)
    assert not out['failed'].any()
    for i in range(200):
        s = pf_ref.solve_newton(tree, np.r_[0.0, p[i]], np.r_[0.0, q[i]])
        assert np.max(np.abs(out['V'][i] - np.sqrt(s['v']))) <= 1e-8, i
        assert np.max(np.abs(out['P'][i] - s['P'][1:])) <= 1e-8, i
        assert np.max(np.abs(out['Q'][i] - s['Q'][1:])) <= 1e-8, i
        assert np.max(np.abs(np.sqrt(out['Isq'][i]) - np.sqrt(s['ell'][1:]))) <= 1e-7, i


def _profiles(net, T=1500, seed=3):
    from flexgpu.network import Network
    from flexgpu.profiles import synthetic_profiles
    return synthetic_profiles(Network(net), len(net['buildings']), T=T, seed=seed)


@pytest.mark.parametrize("name", list(F.CATALOGUE))
def test_ref_env_runs_an_episode_on_every_feeder(name):
    """RefFlexEnv takes any radial feeder: an episode up to the limit, with the mirror's rewards to 1e-6 relative."""
    net = F.feeder(name)
    args = F.env_args(net)
    args.pop("kernel_variant")
    prof = _profiles(net).as_dict()
    na, nb = len(net['buildings']), len(net['bus_numbers'])
    ref = env_ref.RefFlexEnv(args, net=net, profiles=prof, rng=np.random.RandomState(4))
    assert ref.get_state().shape == (3 * nb + 2 * na + 1,) and len(ref.get_obs()) == na
    fon = c_mirror.make_net(ieee33.tree_arrays(net), args, net['buildings'])
    mb = c_mirror.MirrorBatch(fon, prof, 1)
    d = ref._last_reset_draw
    mb.reset(np.array([d['start']]), d['e0'][None], d['a0'][None])
    assert np.max(np.abs(ref._get_bus_v() - mb.V[0])) < 1e-8
    rng = np.random.default_rng(5)
    for t in range(ref.episode_limit - 1):
        a = rng.uniform(0, 1, 4 * na)
        r, done, info = ref.step(a)
        rr, dd, ii = mb.step(a[None])
        assert abs(r - rr[0]) <= 1e-6 * abs(r) + 1e-12, (t, r, rr[0])
        assert done == bool(dd[0]), t
        assert np.max(np.abs(ref._get_bus_v() - mb.V[0])) < 1e-8, t
        if done:
            break
    assert done and ref.steps == ref.episode_limit
