"""Feeder catalogue for the run-time-topology tests, and helpers shared by the GPU parity tests.

Every entry is the reference's network dict (utils/create_net.py:27-38 layout) of a radial feeder other than the
built-in IEEE-33 case with its five buildings, together with the thread-kernel instantiation it is meant to reach.
Which instantiation a feeder gets is not read back from the library: `tree_counts` ports the host's chain / slot
derivation (derive_tree_tables in safe-marl_b200/csrc/flex_common.cuh, on the DFS lane order of build_topology in
flex_api.cu) and `thread_shape` its selection rule (thread_shape_of), and the CPU tests pin each entry to its row.

    name             buses / agents  reaches
    two_bus           2 / 1          nl = 1
    chain33          33 / 5          depth 31 (every pointer-jumping round of the warp sweep), RtShape with na = 5
    limits_16x8      25 / 5          exactly 16 chains and 8 slots (the thread variant's limits)
    slack_star       20 / 2          7 lines leaving the slack bus, each a short chain
    ieee33_4agents   33 / 4          the IEEE-33 tree under RtShape, nl = 32
    ieee33_permuted  33 / 5          shuffled bus_numbers, lines given (to, from): RtShape at nl = 32
    ieee33_rescaled  33 / 5          IEEE-33 shape, impedances x1.7, loads x0.55, no line ratings: static shape,
                                     any_imax = 0
    custom14         14 / 3          two slack lines, two laterals on one bus, a nested lateral
    over_17_chains   26 / 5          17 chains: rejected by the thread variant, run by the warp variant
    over_9_slots     20 / 5          9 slots: rejected by the thread variant, run by the warp variant
"""
import numpy as np

from oracle import env_ref, ieee33

SHAPE_RUNTIME, SHAPE_IEEE33 = "RtShape", "Ieee33"
MAX_SLOTS, MAX_CHAINS = 8, 16                     # FP_MAX_SLOTS, FP_MAX_CHAINS


def make_network(lines, loads, buildings, imax_a=150.0, bus_numbers=None, args=None):
    """The reference's network dict from (FROM, TO, R ohm, X ohm) lines and {bus: (kW, kvar)} loads, converted to per
    unit as create_net.py:17-24 does.  imax_a: rating in ampere of every line (0: none)."""
    a = args or env_ref.DEFAULT_ARGS
    zbase = a["v_nom"] ** 2 * 1000 / a["s_nom"]
    ibase = a["s_nom"] / a["v_nom"]
    nodes = list(bus_numbers) if bus_numbers is not None else \
        sorted({1} | {f for f, _, _, _ in lines} | {t for _, t, _, _ in lines})
    return {
        'bus_numbers': nodes,
        'line_connections': [(f, t) for (f, t, _, _) in lines],
        'line_resistances': {(f, t): r / zbase for (f, t, r, _) in lines},
        'line_reactances': {(f, t): x / zbase for (f, t, _, x) in lines},
        'max_line_currents': {(f, t): imax_a / ibase for (f, t, _, _) in lines},
        'bus_types': {n: (1 if n == 1 else 0) for n in nodes},
        'active_power_demand': {n: loads.get(n, (0, 0))[0] / a["s_nom"] for n in nodes},
        'reactive_power_demand': {n: loads.get(n, (0, 0))[1] / a["s_nom"] for n in nodes},
        'buildings': list(buildings), 'PVs_at_buildings': list(buildings), 'ESSs_at_buildings': list(buildings),
    }


def _uniform_loads(lines, kw, kvar):
    return {t: (kw, kvar) for (_, t, _, _) in lines}


def _two_bus():
    lines = [(1, 2, 6.0, 4.0)]
    return make_network(lines, {2: (900, 400)}, [2])


def _chain33():
    lines = [(i, i + 1, .12 + .004 * i, .06 + .002 * i) for i in range(1, 33)]
    return make_network(lines, _uniform_loads(lines, 72, 32), [33, 9, 2, 25, 17])


def _limits_lines():
    """Trunk 1-2-...-9 with one single-bus lateral on each of buses 2..8 (7 slots), three children on bus 9 (slot 8),
    and six more lines leaving the slack bus: 1 + 7 + 2 + 6 = 16 chains."""
    lines = [(i, i + 1, .40, .25) for i in range(1, 9)]
    nxt = 10
    for b in range(2, 9):
        lines.append((b, nxt, .40, .25)); nxt += 1
    for _ in range(3):
        lines.append((9, nxt, .35, .20)); nxt += 1
    for _ in range(6):
        lines.append((1, nxt, .30, .18)); nxt += 1
    return lines, nxt                                 # nxt: the next free bus number (26)


def _limits_16x8():
    lines, _ = _limits_lines()
    return make_network(lines, _uniform_loads(lines, 140, 60), [9, 12, 20, 25, 4])


def _over_17_chains():
    lines, nxt = _limits_lines()
    lines = lines + [(1, nxt, .30, .18)]             # a seventh extra line leaving the slack bus: 17 chains
    return make_network(lines, _uniform_loads(lines, 140, 60), [9, 12, 20, 26, 4])


def _over_9_slots():
    """Trunk 1-2-...-10, a lateral on each of buses 2..9 and two children on bus 10: 9 branching buses, 10 chains."""
    lines = [(i, i + 1, .25, .15) for i in range(1, 10)]
    nxt = 11
    for b in range(2, 10):
        lines.append((b, nxt, .40, .25)); nxt += 1
    for _ in range(2):
        lines.append((10, nxt, .35, .20)); nxt += 1
    return make_network(lines, _uniform_loads(lines, 240, 105), [10, 13, 20, 5, 18])


def _slack_star():
    lines, nxt = [], 2
    for length in (3, 2, 4, 1, 3, 2, 4):
        prev = 1
        for _ in range(length):
            lines.append((prev, nxt, .35 + .01 * nxt, .20 + .005 * nxt)); prev = nxt; nxt += 1
    return make_network(lines, _uniform_loads(lines, 1250, 560), [8, 20])


def _ieee33(buildings, scale_z=1.0, imax=True, bus_numbers=None, flip=(), scale_load=1.0):
    net = ieee33.create_network(buildings=buildings)
    lines = []
    for (f, t) in net['line_connections']:
        key = (t, f) if (f, t) in flip else (f, t)
        lines.append(key)
    out = dict(net)
    out['line_connections'] = lines
    src = lambda d: {((t, f) if (f, t) in flip else (f, t)): d[(f, t)] for (f, t) in net['line_connections']}
    out['line_resistances'] = {k: v * scale_z for k, v in src(net['line_resistances']).items()}
    out['line_reactances'] = {k: v * scale_z for k, v in src(net['line_reactances']).items()}
    out['max_line_currents'] = {k: (v if imax else 0.0) for k, v in src(net['max_line_currents']).items()}
    out['active_power_demand'] = {b: v * scale_load for b, v in net['active_power_demand'].items()}
    out['reactive_power_demand'] = {b: v * scale_load for b, v in net['reactive_power_demand'].items()}
    if bus_numbers is not None:
        out['bus_numbers'] = list(bus_numbers)
    return out


def _ieee33_permuted():
    perm = list(range(2, 34))
    np.random.default_rng(1).shuffle(perm)
    flip = {(2, 3), (6, 26), (19, 20), (12, 13), (32, 33), (3, 23)}
    return _ieee33([5, 10, 15, 20, 25], bus_numbers=[1] + perm, flip=flip)


# name -> (builder, counts the host must derive, thread shape, thread variant accepts it)
CATALOGUE = {
    "two_bus": (_two_bus, dict(nb=2, na=1, chains=1, slots=0, depth=0), SHAPE_RUNTIME, True),
    "chain33": (_chain33, dict(nb=33, na=5, chains=1, slots=0, depth=31), SHAPE_RUNTIME, True),
    "limits_16x8": (_limits_16x8, dict(nb=25, na=5, chains=16, slots=8, depth=8), SHAPE_RUNTIME, True),
    "slack_star": (_slack_star, dict(nb=20, na=2, chains=7, slots=0, depth=3), SHAPE_RUNTIME, True),
    "ieee33_4agents": (lambda: _ieee33([5, 10, 15, 20]), dict(nb=33, na=4, chains=4, slots=3, depth=16),
                       SHAPE_RUNTIME, True),
    "ieee33_permuted": (_ieee33_permuted, dict(nb=33, na=5, chains=4, slots=3, depth=16), SHAPE_RUNTIME, True),
    "ieee33_rescaled": (lambda: _ieee33([5, 10, 15, 20, 25], scale_z=1.7, imax=False, scale_load=0.55),
                        dict(nb=33, na=5, chains=4, slots=3, depth=16), SHAPE_IEEE33, True),
    "custom14": (lambda: custom14(), dict(nb=14, na=3, chains=6, slots=3, depth=4), SHAPE_RUNTIME, True),
    "over_17_chains": (_over_17_chains, dict(nb=26, na=5, chains=17, slots=8, depth=8), SHAPE_RUNTIME, False),
    "over_9_slots": (_over_9_slots, dict(nb=20, na=5, chains=10, slots=9, depth=9), SHAPE_RUNTIME, False),
}


def feeder(name):
    """The network dict of catalogue entry `name` (a fresh copy)."""
    return CATALOGUE[name][0]()


def variants(name):
    """Kernel variants that accept the feeder."""
    return ("thread", "warp") if CATALOGUE[name][3] else ("warp",)


def cases():
    """(feeder, variant) pairs the library accepts, as pytest parameters."""
    return [(f, v) for f in CATALOGUE for v in variants(f)]


def env_args(net, variant="thread", **extra):
    """The env arguments for `net`: the reference's defaults with its buildings."""
    a = dict(env_ref.DEFAULT_ARGS)
    b = list(net['buildings'])
    a.update(buildings=b, pv_nodes=b, ess_nodes=b, kernel_variant=variant, **extra)
    return a


# ------------------------------------------------------------------ the 14-bus feeder of the first custom-feeder test
#        1 ---- 2 ---- 3 ---- 4 ---- 5
#        |      |\            |
#        |      | 8 -- 9      6 -- 7
#        |      10             \
#        |                      13
#        11 -- 12 -- 14
CUSTOM14_LINES = [(1, 2, .30, .20), (2, 3, .45, .25), (3, 4, .40, .30), (4, 5, .80, .60), (4, 6, .50, .35),
                  (6, 7, .90, .70), (2, 8, .35, .15), (8, 9, .60, .45), (2, 10, .55, .40), (1, 11, .25, .12),
                  (11, 12, .70, .50), (6, 13, .65, .20), (12, 14, .95, .85)]
CUSTOM14_LOADS = {2: (120, 60), 3: (90, 40), 4: (200, 90), 5: (150, 70), 6: (60, 30), 7: (210, 100), 8: (100, 50),
                  9: (80, 30), 10: (140, 60), 11: (60, 20), 12: (300, 150), 13: (75, 35), 14: (180, 80)}
CUSTOM14_BUILDINGS = [5, 9, 14]


def custom14():
    return make_network(CUSTOM14_LINES, CUSTOM14_LOADS, CUSTOM14_BUILDINGS, bus_numbers=list(range(1, 15)))


# ------------------------------------------------------------------ the host's derivation, ported
def lane_parents(parent):
    """build_topology's DFS pre-order (children in ascending bus position) -> parent lane of every lane (-1: the
    slack bus), and the lane of every non-slack bus position."""
    parent = [int(p) for p in parent]
    nb = len(parent)
    kids = {i: [] for i in range(nb)}
    for b in range(1, nb):
        kids[parent[b]].append(b)
    order, stack = [], list(reversed(kids[0]))
    while stack:
        b = stack.pop()
        order.append(b)
        stack += list(reversed(kids[b]))
    lane = {b: k for k, b in enumerate(order)}
    return [lane[parent[b]] if parent[b] > 0 else -1 for b in order], lane


def tree_counts(parent):
    """derive_tree_tables' chain and slot counts, and the depth (most ancestor lines of any line), for a bus-order
    parent array.  A chain starts at lane 0 and at every lane whose parent is not the lane before it; a slot belongs
    to every lane with a child two or more lanes further on."""
    par, _ = lane_parents(parent)
    nl = len(par)
    chains = sum(1 for k in range(nl) if k == 0 or par[k] != k - 1)
    slots = sum(1 for a in range(nl) if any(par[j] == a for j in range(a + 2, nl)))
    depth = 0
    for k in range(nl):
        d, p = 0, par[k]
        while p >= 0:
            d, p = d + 1, par[p]
        depth = max(depth, d)
    return dict(chains=chains, slots=slots, depth=depth)


def _ieee33_lane_tables():
    """Ieee33Tree::PAR / COL of flex_common.cuh, from the built-in feeder."""
    t = ieee33.tree_arrays(ieee33.create_network())
    par, lane = lane_parents(t['parent'])
    col = [None] * len(par)
    for b, k in lane.items():
        col[k] = b - 1
    return par, col


def thread_shape(net):
    """thread_shape_of plus build_topology's agent rule: the static IEEE-33 instantiation for the built-in tree (same
    DFS parents and dataset columns) with five agents, RtShape for anything else."""
    t = ieee33.tree_arrays(net)
    par, lane = lane_parents(t['parent'])
    col = [None] * len(par)
    for b, k in lane.items():
        col[k] = b - 1
    ipar, icol = _ieee33_lane_tables()
    same = par == ipar and col == icol
    return SHAPE_IEEE33 if same and len(net['buildings']) == 5 else SHAPE_RUNTIME


# ------------------------------------------------------------------ safety maps
def lindistflow_map(tree):
    """LinDistFlow sensitivities of any radial tree: V = A [P_1, Q_1, ..., P_nb, Q_nb] + 1 with dV_n / dP_m = -sum R_l
    and dV_n / dQ_m = -sum X_l over the lines shared by the root paths of buses n and m (lines named by their far bus)."""
    parent, R, X = np.asarray(tree["parent"]), np.asarray(tree["R"]), np.asarray(tree["X"])
    nb = len(parent)
    path = []
    for n in range(nb):
        p, s = n, set()
        while parent[p] >= 0:
            s.add(p); p = parent[p]
        path.append(s)
    A = np.zeros((nb, 2 * nb))
    for n in range(nb):
        for m in range(nb):
            shared = list(path[n] & path[m])
            A[n, 2 * m] = -R[shared].sum(); A[n, 2 * m + 1] = -X[shared].sum()
    return A, np.ones(nb)


def ref_stub(net, args, state_row):
    """A RefFlexEnv-shaped object carrying one GPU env's current values (what safety_ref.parse_actions reads), from its
    fp64 get_state row [P(nb), Q(nb), Ppv(na), V(nb), price, E(na)]."""
    nb, na = len(net['bus_numbers']), len(net['buildings'])
    st = state_row
    ref = env_ref.RefFlexEnv.__new__(env_ref.RefFlexEnv)
    ref.args = env_ref._Args(dict(env_ref.DEFAULT_ARGS)); ref.args.update(args)
    ref.base_powergrid = net
    ref.current_active_demand = {b: float(st[i]) for i, b in enumerate(net['bus_numbers'])}
    ref.current_reactive_demand = {b: float(st[nb + i]) for i, b in enumerate(net['bus_numbers'])}
    ref.current_pv_power = {b: float(st[2 * nb + i]) for i, b in enumerate(net['PVs_at_buildings'])}
    ref.current_ess_energy = {b: float(st[3 * nb + na + 1 + i]) for i, b in enumerate(net['ESSs_at_buildings'])}
    return ref


# ------------------------------------------------------------------ handle state snapshots
def snapshot(env):
    """Every byte of the handle's per-env state a step can write, and the statistics partials' sums."""
    import torch
    torch.cuda.synchronize()
    ring = env.obs_ring()
    pf, qf, isq = env.line_flows
    out = {"rec": env.rec.clone(), "V": env.voltages.clone(), "setp": env.setpoints.clone(),
           "hist": env._history(False).clone(), "ring": ring.ring.clone(), "slot": ring.slot}
    if pf is not None:
        out.update(pf=pf.clone(), qf=qf.clone(), isq=isq.clone())
    out["stats"] = {k: v.clone() for k, v in env.episode_stats(reduce=False).items()}
    torch.cuda.synchronize()
    return out


def assert_same_bytes(a, b):
    import torch
    assert a.keys() == b.keys()
    for k in a:
        if k == "stats":
            for s in a[k]:
                assert torch.equal(a[k][s].view(torch.int64), b[k][s].view(torch.int64)), s
        elif isinstance(a[k], torch.Tensor):
            x, y = a[k], b[k]
            if x.dtype == torch.float64:
                x, y = x.view(torch.int64), y.view(torch.int64)     # bits, NaN included
            assert torch.equal(x, y), k
        else:
            assert a[k] == b[k], k
