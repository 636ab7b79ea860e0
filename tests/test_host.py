"""CPU: host-side logic of the product package (no GPU): network parsing, configuration,
profile generation.  Cross-checked against the oracle's independent restatement."""
import numpy as np
import pytest

from flexgpu.config import DEFAULT_ENV_ARGS, make_fp_config, normalize_args
from flexgpu.network import Network, create_network
from flexgpu.profiles import Profiles, synthetic_profiles


def test_create_network_matches_oracle_restatement(net):
    mine = create_network(DEFAULT_ENV_ARGS)
    assert set(mine) == set(net)                                     # utils/create_net.py:27-38 keys
    for k in ('bus_numbers', 'buildings', 'PVs_at_buildings', 'ESSs_at_buildings'):
        assert list(mine[k]) == list(net[k])
    assert set(mine['line_connections']) == set(net['line_connections'])
    for k in ('line_resistances', 'line_reactances', 'max_line_currents', 'active_power_demand',
              'reactive_power_demand', 'bus_types'):
        assert mine[k] == net[k]


def test_network_positions_and_parents(network, tree):
    assert network.n_bus == 33 and network.parent[0] == -1
    assert np.array_equal(network.parent, tree['parent'])
    assert np.array_equal(network.r, tree['R']) and np.array_equal(network.x, tree['X'])
    assert network.position[19] == 18 and network.parent[18] == 1      # bus 19 hangs off bus 2
    assert network.parent[network.position[26]] == network.position[6]


def test_network_rejects_non_radial_or_misplaced_slack():
    net = create_network(DEFAULT_ENV_ARGS)
    bad = dict(net); bad['line_connections'] = net['line_connections'] + [(18, 33)]
    for key in ('line_resistances', 'line_reactances', 'max_line_currents'):
        bad[key] = dict(net[key]); bad[key][(18, 33)] = 0.01
    with pytest.raises(ValueError):
        Network(bad)
    bad = dict(net); bad['bus_numbers'] = net['bus_numbers'][1:] + [1]
    with pytest.raises(ValueError):
        Network(bad)


def test_fp_config_values(network):
    a = normalize_args({"alg": "safemaddpg"})
    c = make_fp_config(a, network)
    assert c.n_bus == 33 and c.n_agents == 5 and c.raw_actions == 1
    assert c.kappa == float.fromhex('0x1.509290e9d53d5p-2') and c.delta_t == 0.25
    assert list(c.agent_bus) == [4, 9, 14, 19, 24] and c.parent[0] == -1 and c.parent[18] == 1
    assert make_fp_config(normalize_args(None), network).raw_actions == 0
    with pytest.raises(ValueError):
        make_fp_config(normalize_args({"pv_nodes": [5, 10]}), network)      # quirk Q8 guard


def test_namedtuple_args_are_accepted():
    from flexgpu.config import convert
    a = normalize_args(convert({"history": 12, "seed": 3}))
    assert a["history"] == 12 and a["seed"] == 3 and a["episode_limit"] == 96


def test_synthetic_profiles_shape_and_range(network):
    p = synthetic_profiles(network, 5, T=960, seed=0)
    assert p.P.shape == (960, 32) and p.Q.shape == (960, 32) and p.PV.shape == (960, 5) and p.price.shape == (960,)
    assert p.P.dtype == np.float64 and p.P.flags.c_contiguous
    assert p.PV.min() >= 0 and p.PV.max() <= 0.15 and np.all(p.PV[0:20] == 0)       # night
    assert 0.05 <= p.price.min() and p.price.max() <= 0.30
    ratio = p.P.mean(axis=0) / network.base_p[1:]
    assert np.all(ratio > 0.3) and np.all(ratio < 1.05)
    q = synthetic_profiles(network, 5, T=960, seed=0)
    assert np.array_equal(p.P, q.P) and p.n_days() == 9


def test_profiles_validation():
    with pytest.raises(ValueError):
        Profiles(np.zeros((10, 32)), np.zeros((9, 32)), np.zeros((10, 5)), np.zeros(10))


def test_translate_action_matches_reference_function():
    """utils/util.py::translate_action itself produced the fixture (tests/golden/make_ref_golden.py):
    the numpy restatement used by the mirror and flexgpu.util.translate_action reproduce it bit for bit."""
    import os
    from collections import namedtuple
    import numpy as np
    import torch
    from oracle import c_mirror
    from flexgpu import translate_action, prep_obs
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_translate_action.npz"))
    lo, hi = float(g["low"][0]), float(g["high"][0])
    assert np.array_equal(c_mirror.translate_action_f32(g["x"], lo, hi).reshape(g["y"].shape), g["y"])
    A = namedtuple("A", "continuous action_low action_high")(True, lo, hi)
    for i in (0, 1, 63):
        raw, cp = translate_action(A, torch.from_numpy(g["x"][i]), None)
        assert cp.dtype == torch.float32 and np.array_equal(cp.numpy(), g["y"][i])
    assert g["y"].min() >= 0.5 and g["y"].max() <= 1.0                                   # quirk Q5
    obs = [np.arange(144, dtype=np.float64) + i for i in range(5)]
    t = prep_obs(obs)
    assert t.dtype == torch.float32 and tuple(t.shape) == (5, 144)
    assert prep_obs(torch.zeros(7, 5, 144, dtype=torch.float64)).shape == (7, 5, 144)


def test_bench_reference_arm_runs_on_cpu():
    """`bench.py --impl reference` (the CPU arm the driver launches next to the GPU arm) needs no GPU:
    one JSON line with the contract's keys, the same metric / unit / workload naming as the GPU arm."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--envs-per-gpu", "2048", "--rows", "3000"], capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "env-steps/s" and line["higher_is_better"] is True
    assert line["metric"] == "33-bus env-steps/sec (incl. power flow)" and line["value"] > 0
    assert line["config"]["workload"].startswith("fused_env_step_2048_envs_per_gpu")
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]


@pytest.mark.parametrize("extra,message", [(["--steps", "0"], "--steps must be at least 1"),
                                           (["--impl", "reference", "--dump-outputs", "out"], "does not apply to --impl reference")])
def test_bench_rejects_arguments_it_cannot_honour(extra, message):
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py")] + extra, capture_output=True, text=True, timeout=60, cwd=root)
    assert out.returncode == 2 and message in out.stderr, out.stderr[-2000:]


# ---------------------------------------------------------------------------------------------------
def test_load_csv_profiles_equals_the_reference_loaders(tmp_path):
    """flexgpu.load_csv_profiles against the output of the reference's own _load_*_data + resample_data
    (flexibility_provision_env.py:431-471), which parsed the SAME csv text (tests/golden/make_ref_golden.py):
    5-minute load / PV rows with missing stretches and hourly prices -> 15-minute means, up-sampling, linear
    interpolation, the three scale factors."""
    import os
    from flexgpu.profiles import csv_profiles_available, load_csv_profiles
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_loaders.npz"))
    assert not csv_profiles_available(str(tmp_path))
    for name in ("pv_active", "load_active", "load_reactive", "prices"):
        (tmp_path / f"{name}.csv").write_bytes(g["csv_" + name].tobytes())
    assert csv_profiles_available(str(tmp_path))
    args = dict(sample_interval="15min", demand_scale=float(g["demand_scale"][0]),
                reactive_scale=float(g["reactive_scale"][0]), pv_scale=float(g["pv_scale"][0]))
    prof = load_csv_profiles(str(tmp_path), args)
    T = prof.T
    assert T == min(len(g["P"]), len(g["price"])) and prof.time_delta == int(g["time_delta"][0])
    assert np.array_equal(prof.P, g["P"][:T]) and np.array_equal(prof.Q, g["Q"][:T])
    assert np.array_equal(prof.PV, g["PV"][:T]) and np.array_equal(prof.price, g["price"][:T])
    assert not np.isnan(prof.P).any() and prof.n_days() >= int(g["pv_days"][0]) - 1
    # the gap of a whole hour was filled by interpolation, the hourly prices were up-sampled
    assert np.all(np.diff(prof.price[:5]) != 0)


def test_lfs_pointer_is_not_mistaken_for_data(tmp_path):
    from flexgpu.profiles import CSV_NAMES, csv_profiles_available
    for n in CSV_NAMES:
        (tmp_path / n).write_text("version https://git-lfs.github.com/spec/v1\noid sha256:0\nsize 1\n")
    assert not csv_profiles_available(str(tmp_path))
